// Per-residue mode (plotsomefastas, plaac.java:610-647), throughput version.
//
// The two posterior columns need the ABSOLUTE forward and backward variables of the lookup-table recurrences in the
// reference's operation order (exp((a+b) - lpseq), posteriorl :3349-3411): the LUT error accumulates along the
// sequence, so there is no associative shortcut that reproduces the jar to 1e-9.  Each recurrence therefore stays
// one sequential chain per protein (lane = protein on the length-bucketed stream, as in the summary kernels) and the
// mode is organised around memory traffic instead:
//
//   k_res_vit     Viterbi max-plus recurrence (viterbidecodel :3077-3121), traceback bits, SWAR traceback -> Viterbi
//                 bits, one 32-bit word per 16 residues per lane
//   k_res_bwd     backward recurrence (:3378-3391) -> scratch planes B0/B1 in the bucketed layout
//                 [slot][residue-in-slot][lane]: every warp store is one 256-byte line
//   k_res_fwd     forward recurrence (:3356-3367) -> scratch planes A0/A1, same layout.  The three recurrences are
//                 independent chains and run concurrently on three streams
//   k_res_lpseq   lpseq per protein (:3393-3396)
//   k_res_post    fully parallel, one warp per 16-residue x 32-protein slot: pp = exp((a+b) - lpseq) (:3401-3405) and
//                 the MAP bit (mapdecodel :4032-4045); tiles are transposed through shared memory and written
//                 protein-major as 128-byte runs
//   k_res_bits    Viterbi/MAP bit words -> one byte per residue, protein-major, coalesced
//   k_res_tracks  the eight disorderreport tracks (:4866-4903, slidingaverage :2585-2662) from fp64 prefix sums: one
//                 warp per protein walks tiles of 256 consecutive residues (+2w halo each side); pass-1 window sums
//                 are differences of a prefix sum of per-residue values, pass-2 sums are differences of a prefix sum
//                 of the pass-1 sums (sum-of-window-sums identity).  All loads and stores are coalesced.
//
// Scratch traffic: 32 B/aa written and read once; output 82 B/aa.
#pragma once
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "residue_kernel.cuh"
#include "summary_kernel_v2.cuh"

namespace plaac {

constexpr int kResThreads = 256;   // k_res_vit, k_res_bits
constexpr int kResPostThreads = 128;
constexpr int kResHmmThreads = 512;  // k_res_bwd, k_res_fwd (one 64 KB LUT per CTA)
constexpr uint32_t kResOffLe = 0;                                     // double2 [32 codes][8 lane copies] {le0, le1}
constexpr uint32_t kResOffLut2 = 4096;                                // double2 [4002]
constexpr uint32_t kResFixedBytes = kResOffLut2 + (PLAAC_LUT_LEN + 1) * 16;
constexpr int kTilePitch = 33;                                        // doubles per tile row (conflict-free transpose)
constexpr uint32_t kResTileBytes = 2 * 16 * kTilePitch * 8;           // per warp: two 16 x 32 tiles

struct ResArgs {
    BatchView bv;
    KScalars ks;
    const DeviceTables* tabs;
    plaac_residue_out out;
    int64_t res_base;    // residue index of out.*[0]
    double* B0;          // backward variables, bucketed layout [slot][residue in slot][lane]
    double* B1;
    double* A0;          // forward variables, same layout
    double* A1;
    uint32_t* mapw;      // MAP bits, one word per slot per lane
    double* lpseq;       // per rank
};

__device__ __forceinline__ void res_stage_tables(unsigned char* sm, const DeviceTables* T)
{
    double2* lut2 = reinterpret_cast<double2*>(sm + kResOffLut2);
    for (int i = threadIdx.x; i <= PLAAC_LUT_LEN; i += blockDim.x) {
        const double l0 = i < PLAAC_LUT_LEN ? T->lut[i] : 0.0;
        const double l1 = i + 1 < PLAAC_LUT_LEN ? T->lut[i + 1] : 0.0;
        lut2[i] = make_double2(l0, l1);
    }
    double2* le = reinterpret_cast<double2*>(sm + kResOffLe);
    for (int i = threadIdx.x; i < 32 * 8; i += blockDim.x) le[i] = make_double2(T->le0[i >> 3], T->le1[i >> 3]);
    __syncthreads();
}

struct LaneView {
    int n;
    int32_t prot;
    int64_t cb;
    int nch;
    int64_t base;  // residue 0 of the protein in the output arrays
};

__device__ __forceinline__ LaneView lane_view(const BatchView& bv, int64_t b, int lane, int64_t res_base)
{
    LaneView v;
    const int64_t rank = b * 32 + lane;
    v.n = 0;
    v.prot = -1;
    v.base = 0;
    if (rank < bv.nprot) {
        v.prot = bv.order[rank];
        const int64_t o = bv.offsets[v.prot];
        v.n = (int)eff_len(bv.offsets[v.prot + 1] - o, bv.long_min);  // long proteins: long_residue.cuh
        v.base = o - res_base;
    }
    v.cb = bv.chunk_base[b];
    v.nch = (int)(bv.chunk_base[b + 1] - v.cb);
    return v;
}

__device__ __forceinline__ uint32_t word_of(const uint4& v, int q)
{
    return q == 0 ? v.x : q == 1 ? v.y : q == 2 ? v.z : v.w;
}

// ------------------------------------------------------------------------------------------------ Viterbi
__global__ void __launch_bounds__(kResThreads) k_res_vit(ResArgs g)
{
    __shared__ double2 le_s[32][8];
    for (int i = threadIdx.x; i < 32 * 8; i += blockDim.x) le_s[i >> 3][i & 7] = make_double2(g.tabs->le0[i >> 3], g.tabs->le1[i >> 3]);
    __syncthreads();
    const KScalars& ks = g.ks;
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < g.bv.nbuckets; b += warps) {
        const LaneView L = lane_view(g.bv, b, lane, g.res_base);
        const int n = L.n;
        const uint4* sp = g.bv.stream + L.cb * 32 + lane;
        uint32_t* tbp = g.bv.tbw + L.cb * 32 + lane;
        double s0 = 0, s1 = 0;
        uint32_t acc0 = 0, acc1 = 0;
        uint4 nxt = L.nch > 0 ? sp[0] : make_uint4(0, 0, 0, 0);
        for (int j = 0; j < L.nch; j++) {
            const uint4 cw = nxt;
            if (j + 1 < L.nch) nxt = sp[(size_t)(j + 1) * 32];
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int t = 16 * j + i;
                const uint32_t cd = (word_of(cw, i >> 2) >> ((i & 3) * 8)) & 31u;
                const double2 le = le_s[cd][lane & 7];
                uint32_t tb0u = 0, tb1u = 0;
                if (t < n) {
                    if (t == 0) {
                        s0 = ks.li0 + le.x;
                        s1 = ks.li1 + le.y;
                    } else {
                        const double v00 = ks.lt00 + s0, v10 = ks.lt10 + s1;
                        const double v01 = ks.lt01 + s0, v11 = ks.lt11 + s1;
                        const bool tb0 = v10 > v00, tb1 = v11 > v01;
                        s0 = (tb0 ? v10 : v00) + le.x;
                        s1 = (tb1 ? v11 : v01) + le.y;
                        tb0u = tb0;
                        tb1u = tb1;
                    }
                }
                acc0 = __funnelshift_r(acc0, tb0u, 1);
                acc1 = __funnelshift_r(acc1, tb1u, 1);
            }
            tbp[(size_t)j * 32] = __byte_perm(acc0, acc1, 0x7632);
        }
        if (n < 1) continue;
        // traceback (:3102-3113) as a suffix scan of 2->2 maps per 16-residue word (see summary_kernel_v2.cuh)
        int v = (s1 + ks.lf1 > s0 + ks.lf0) ? 1 : 0;
        const int jlast = (n - 1) >> 4;
        uint32_t tw_next = tbp[(size_t)jlast * 32];
        for (int j = jlast; j >= 0; j--) {
            const uint32_t tw = tw_next;
            if (j > 0) tw_next = tbp[(size_t)(j - 1) * 32];
            const int hi = (j == jlast) ? ((n - 1) & 15) : 15;
            const uint32_t valid = (2u << hi) - 1u, below = valid >> 1;
            const uint32_t P0 = tw & 0xffffu, P1 = tw >> 16;
            uint32_t A0 = (P0 >> 1) & below;
            uint32_t A1 = ((P1 >> 1) & below) | (0xffffu & ~below);
#pragma unroll
            for (int sft = 1; sft < 16; sft <<= 1) {
                const uint32_t B0 = A0 >> sft;
                const uint32_t B1 = (A1 >> sft) | (0xffffu & ~(0xffffu >> sft));
                const uint32_t n0 = (B0 & A1) | (~B0 & A0);
                const uint32_t n1 = (B1 & A1) | (~B1 & A0);
                A0 = n0;
                A1 = n1;
            }
            const uint32_t vb = (v ? A1 : A0) & valid;
            v = (int)(((vb & 1u) ? P1 : P0) & 1u);
            tbp[(size_t)j * 32] = vb;
        }
    }
}

// ------------------------------------------------------------------------------------------------ backward
__global__ void __launch_bounds__(kResHmmThreads) k_res_bwd(ResArgs g)
{
    extern __shared__ __align__(16) unsigned char res_smem[];
    res_stage_tables(res_smem, g.tabs);
    const uint32_t sbase = smem_u32(res_smem);
    const KScalars& ks = g.ks;
    const int lane = threadIdx.x & 31;
    const uint32_t le_base = sbase + kResOffLe + (uint32_t)(lane & 7) * 16u;
    const uint32_t lut_addr = sbase + kResOffLut2;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < g.bv.nbuckets; b += warps) {
        const LaneView L = lane_view(g.bv, b, lane, g.res_base);
        const int n = L.n;
        const uint4* sp = g.bv.stream + L.cb * 32 + lane;
        double* B0 = g.B0 + (size_t)L.cb * 512 + lane;
        double* B1 = g.B1 + (size_t)L.cb * 512 + lane;
        double b0 = 0, b1 = 0;
        uint32_t cnext = 0;  // code of residue t+1
        uint4 nxt = L.nch > 0 ? sp[(size_t)(L.nch - 1) * 32] : make_uint4(0, 0, 0, 0);
        for (int j = L.nch - 1; j >= 0; j--) {
            const uint4 cw = nxt;
            if (j > 0) nxt = sp[(size_t)(j - 1) * 32];
#pragma unroll
            for (int i = 15; i >= 0; i--) {
                const int t = 16 * j + i;
                const uint32_t cd = (word_of(cw, i >> 2) >> ((i & 3) * 8)) & 31u;
                if (t < n) {
                    if (t == n - 1) {
                        b0 = ks.lf0;  // :3379-3381
                        b1 = ks.lf1;
                    } else {
                        // b[i][t] = LSE_k( (lt[i][k] + b[k][t+1]) + le[k][aa[t+1]] ), k ascending (:3384-3389)
                        const double2 le = lds_v2f64(le_base + (cnext << 7));
                        const double x0 = (ks.lt00 + b0) + le.x, x1 = (ks.lt01 + b1) + le.y;
                        const double y0 = (ks.lt10 + b0) + le.x, y1 = (ks.lt11 + b1) + le.y;
                        b0 = lse_lut2<false>(x0, x1, lut_addr);
                        b1 = lse_lut2<false>(y0, y1, lut_addr);
                    }
                    B0[((size_t)j * 16 + i) * 32] = b0;
                    B1[((size_t)j * 16 + i) * 32] = b1;
                    cnext = cd;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ forward
__global__ void __launch_bounds__(kResHmmThreads) k_res_fwd(ResArgs g)
{
    extern __shared__ __align__(16) unsigned char res_smem[];
    res_stage_tables(res_smem, g.tabs);
    const uint32_t sbase = smem_u32(res_smem);
    const KScalars& ks = g.ks;
    const int lane = threadIdx.x & 31;
    const uint32_t le_base = sbase + kResOffLe + (uint32_t)(lane & 7) * 16u;
    const uint32_t lut_addr = sbase + kResOffLut2;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < g.bv.nbuckets; b += warps) {
        const LaneView L = lane_view(g.bv, b, lane, g.res_base);
        const int n = L.n;
        const uint4* sp = g.bv.stream + L.cb * 32 + lane;
        double* A0 = g.A0 + (size_t)L.cb * 512 + lane;
        double* A1 = g.A1 + (size_t)L.cb * 512 + lane;
        double a0 = 0, a1 = 0;
        uint4 nxt = L.nch > 0 ? sp[0] : make_uint4(0, 0, 0, 0);
        for (int j = 0; j < L.nch; j++) {
            const uint4 cw = nxt;
            if (j + 1 < L.nch) nxt = sp[(size_t)(j + 1) * 32];
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int t = 16 * j + i;
                const uint32_t cd = (word_of(cw, i >> 2) >> ((i & 3) * 8)) & 31u;
                if (t < n) {
                    const double2 le = lds_v2f64(le_base + (cd << 7));
                    if (t == 0) {
                        a0 = ks.li0 + le.x;  // :3356-3358
                        a1 = ks.li1 + le.y;
                    } else {
                        const double f0 = lse_lut2<false>(ks.lt00 + a0, ks.lt10 + a1, lut_addr) + le.x;  // :3359-3367
                        const double f1 = lse_lut2<false>(ks.lt01 + a0, ks.lt11 + a1, lut_addr) + le.y;
                        a0 = f0;
                        a1 = f1;
                    }
                    A0[((size_t)j * 16 + i) * 32] = a0;
                    A1[((size_t)j * 16 + i) * 32] = a1;
                }
            }
        }
    }
}

// lpseq = logeapeb(a[0][0] + b[0][0], a[1][0] + b[1][0]) per protein (:3393-3396); lane = rank
__global__ void __launch_bounds__(256) k_res_lpseq(ResArgs g)
{
    const int64_t rank = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (rank >= g.bv.nprot) return;
    {
        const int32_t prot = g.bv.order[rank];
        if (eff_len(g.bv.offsets[prot + 1] - g.bv.offsets[prot], g.bv.long_min) == 0) {  // no slot to read
            g.lpseq[rank] = 0.0;
            return;
        }
    }
    const size_t at = (size_t)g.bv.chunk_base[rank >> 5] * 512 + (size_t)(rank & 31);
    g.lpseq[rank] = lse_lut_g(g.A0[at] + g.B0[at], g.A1[at] + g.B1[at], g.tabs->lut, g.ks.ln2);
}

// ------------------------------------------------------------------------------------------------ posteriors + MAP
// Fully parallel: one warp per 32-lane slot (16 residues of 32 proteins).  pp = exp((a + b) - lpseq) (:3401-3405),
// MAP bit = pp1 > pp0 (:4036-4040).  The 16 x 32 tiles are transposed through shared memory and written
// protein-major: lanes 0-15 carry 16 consecutive post_bg values of one protein, lanes 16-31 its post_prd values.
__global__ void __launch_bounds__(kResPostThreads) k_res_post(ResArgs g)
{
    __shared__ double tiles[kResPostThreads / 32][2][16 * kTilePitch];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double* tile0 = tiles[wid][0];
    double* tile1 = tiles[wid][1];
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t total = g.bv.chunk_base[g.bv.nbuckets];
    for (int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < total; s += warps) {
        const int64_t b = g.bv.slot_bucket[s];
        const int j = (int)(s - g.bv.chunk_base[b]);
        const int64_t rank = b * 32 + lane;
        int n = 0;
        int64_t base = 0;
        double lpseq = 0;
        if (rank < g.bv.nprot) {
            const int32_t prot = g.bv.order[rank];
            const int64_t o = g.bv.offsets[prot];
            n = (int)eff_len(g.bv.offsets[prot + 1] - o, g.bv.long_min);
            base = o - g.res_base;
            lpseq = g.lpseq[rank];
        }
        const size_t at = (size_t)s * 512 + lane;
        double a0[16], a1[16];
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const bool in = 16 * j + i < n;
            a0[i] = in ? g.A0[at + (size_t)i * 32] + g.B0[at + (size_t)i * 32] : 0.0;
            a1[i] = in ? g.A1[at + (size_t)i * 32] + g.B1[at + (size_t)i * 32] : 0.0;
        }
        uint32_t mapbits = 0;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const double p0 = exp(a0[i] - lpseq), p1 = exp(a1[i] - lpseq);
            if (16 * j + i < n) mapbits |= (p1 > p0 ? 1u : 0u) << i;
            tile0[i * kTilePitch + lane] = p0;
            tile1[i * kTilePitch + lane] = p1;
        }
        g.mapw[(size_t)s * 32 + lane] = mapbits;
        __syncwarp();
        const int half = lane >> 4, ii = lane & 15;
        const double* tsrc = (half ? tile1 : tile0) + ii * kTilePitch;
        double* const dsts = half ? g.out.post_prd : g.out.post_bg;
#pragma unroll 8
        for (int q = 0; q < 32; q++) {
            const int nq = __shfl_sync(0xffffffffu, n, q);
            const int64_t bq = __shfl_sync(0xffffffffu, base, q);
            if (16 * j + ii < nq) dsts[bq + 16 * j + ii] = tsrc[q];
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------ bit words -> bytes
__global__ void __launch_bounds__(kResThreads) k_res_bits(ResArgs g)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int64_t b = blockIdx.x; b < g.bv.nbuckets; b += gridDim.x) {
        const int64_t cb = g.bv.chunk_base[b];
        for (int q = wid; q < 32; q += nw) {
            const int64_t rank = b * 32 + q;
            if (rank >= g.bv.nprot) break;
            const int32_t prot = g.bv.order[rank];
            const int64_t o = g.bv.offsets[prot];
            const int n = (int)eff_len(g.bv.offsets[prot + 1] - o, g.bv.long_min);
            const int64_t base = o - g.res_base;
            const uint32_t* vw = g.bv.tbw + cb * 32 + q;
            const uint32_t* mw = g.mapw + cb * 32 + q;
            // a lane writes four consecutive OUTPUT bytes (one aligned 32-bit store, 128 bytes per warp store); groups
            // are aligned to the output ADDRESS, so the first and last group of a protein may be partial
            auto expand = [&](uint8_t* dst, const uint32_t* words) {
                if (!dst) return;
                const int mis = (int)(reinterpret_cast<uintptr_t>(dst + base) & 3);
                for (int64_t t0l = -mis + 4 * lane; t0l < n; t0l += 128) {
                    const int t0 = (int)t0l;  // -3 .. -1 for a partial first group
                    uint32_t v = 0;
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int t = t0 + k;
                        if (t >= 0 && t < n) v |= ((words[(size_t)(t >> 4) * 32] >> (t & 15)) & 1u) << (8 * k);
                    }
                    if (t0 >= 0 && t0 + 3 < n)
                        *reinterpret_cast<uint32_t*>(dst + base + t0) = v;
                    else {
#pragma unroll
                        for (int k = 0; k < 4; k++)
                            if (t0 + k >= 0 && t0 + k < n) dst[base + t0 + k] = (uint8_t)(v >> (8 * k));
                    }
                }
            };
            expand(g.out.vit, vw);
            expand(g.out.map, mw);
        }
    }
}

// ------------------------------------------------------------------------------------------------ tracks
constexpr int kTrackTile = 256;
constexpr int kTrackWarps = 4;

// inclusive prefix sum of arr[0..len) in place; lane `lane` owns the contiguous run [lane*per, lane*per+per)
template <typename T>
__device__ __forceinline__ void warp_scan_inplace(T* arr, int len, int per, int lane)
{
    const int lo = lane * per, hi = min(lo + per, len);
    T run = 0;
    for (int e = lo; e < hi; e++) {
        run = run + arr[e];
        arr[e] = run;
    }
    T inc = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc = inc + o;
    }
    T ex = __shfl_up_sync(0xffffffffu, inc, 1);  // sum of the runs of the lower lanes
    if (lane == 0) ex = 0;
    if (lane > 0)
        for (int e = lo; e < hi; e++) arr[e] = arr[e] + ex;
    __syncwarp();
}

// the four tracks scanned together: four independent dependency chains per lane instead of one
__device__ __forceinline__ void warp_scan4_inplace(double* a, double* b, double* c, int* d, int len, int per, int lane)
{
    const int lo = lane * per, hi = min(lo + per, len);
    double ra = 0, rb = 0, rc = 0;
    int rd = 0;
    for (int e = lo; e < hi; e++) {
        ra = ra + a[e];
        rb = rb + b[e];
        rc = rc + c[e];
        rd = rd + d[e];
        a[e] = ra;
        b[e] = rb;
        c[e] = rc;
        d[e] = rd;
    }
    double ia = ra, ib = rb, ic = rc;
    int id = rd;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const double oa = __shfl_up_sync(0xffffffffu, ia, s), ob = __shfl_up_sync(0xffffffffu, ib, s);
        const double oc = __shfl_up_sync(0xffffffffu, ic, s);
        const int od = __shfl_up_sync(0xffffffffu, id, s);
        if (lane >= s) {
            ia = ia + oa;
            ib = ib + ob;
            ic = ic + oc;
            id = id + od;
        }
    }
    double ea = __shfl_up_sync(0xffffffffu, ia, 1), eb = __shfl_up_sync(0xffffffffu, ib, 1);
    double ec = __shfl_up_sync(0xffffffffu, ic, 1);
    int ed = __shfl_up_sync(0xffffffffu, id, 1);
    if (lane > 0) {
        for (int e = lo; e < hi; e++) {
            a[e] = a[e] + ea;
            b[e] = b[e] + eb;
            c[e] = c[e] + ec;
            d[e] = d[e] + ed;
        }
    }
    __syncwarp();
}

struct TrackArgs {
    const uint8_t* codes;     // protein-major, 1 byte per residue
    const int64_t* offsets;
    int64_t off_base;         // offsets are relative to this residue index for `codes`
    int64_t res_base;         // ... and to this one for the output arrays
    int64_t nprot;
    KScalars ks;
    const DeviceTables* tabs;
    plaac_residue_out out;
    int nx;                   // kTrackTile + 4w
    int per_x, per_s;         // elements per lane of the two scans (odd: conflict-free)
    // Long proteins (>= long_min residues) are skipped by the protein-per-warp launch and handled by a second launch
    // with long_list set: blockIdx.y picks the protein, the warps of the grid's x dimension share its tiles.
    int64_t long_min;
    const int32_t* long_list;
};

__global__ void __launch_bounds__(kTrackWarps * 32) k_res_tracks(TrackArgs g)
{
    extern __shared__ __align__(16) unsigned char trk_smem[];
    __shared__ double tab_h[32], tab_l[32], tab_p[32];
    for (int i = threadIdx.x; i < 32; i += blockDim.x) {
        tab_h[i] = g.tabs->hyd[i];
        tab_l[i] = g.tabs->llr[i];
        tab_p[i] = g.tabs->pap[i];
    }
    __syncthreads();
    const KScalars& ks = g.ks;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int w = ks.w, full = 2 * w + 1, Wfull = full * full;
    const int NX = g.nx, NS = kTrackTile + 2 * w;
    const double rfull = 1.0 / (double)full, rWfull = 1.0 / (double)Wfull;
    // per-warp arrays; the pass-1 window sums S* (NS <= NX entries) overwrite the prefix sums X* in place, 32 at a
    // time in ascending order (see step 2), which halves the footprint and lets five CTAs share an SM
    const size_t per_warp = (size_t)NX * (3 * 8 + 4) + (size_t)NX + 64;
    unsigned char* base = trk_smem + (size_t)wid * ((per_warp + 15) & ~(size_t)15);
    double* Xh = reinterpret_cast<double*>(base);
    double* Xl = Xh + NX;
    double* Xp = Xl + NX;
    int* Xc = reinterpret_cast<int*>(Xp + NX);
    uint8_t* Cd = reinterpret_cast<uint8_t*>(Xc + NX);
    double *Sh = Xh, *Sl = Xl, *Sp = Xp;
    int* Sc = Xc;

    const int64_t warps = (int64_t)gridDim.x * kTrackWarps;
    const bool by_tile = g.long_list != nullptr;
    for (int64_t it = (int64_t)blockIdx.x * kTrackWarps + wid; it < (by_tile ? warps : g.nprot); it += warps) {
        const int64_t p = by_tile ? (int64_t)g.long_list[blockIdx.y] : it;
        const int64_t o = g.offsets[p];
        const int n = (int)(g.offsets[p + 1] - o);
        if (!by_tile && n >= g.long_min) continue;
        const uint8_t* src = g.codes + (o - g.off_base);
        const int64_t ob = o - g.res_base;
        const int t_first = by_tile ? (int)it * kTrackTile : 0;
        const int64_t t_step = by_tile ? warps * kTrackTile : kTrackTile;
        for (int64_t t0l = t_first; t0l < n; t0l += t_step) {
            const int t0 = (int)t0l;
            const int u_lo = t0 - 2 * w;  // residue of X*[0]
            // the last tile of a protein is shorter: nothing beyond residue n-1 has to be staged or scanned (prefix
            // sums stay constant there; reads clamp to the last element)
            const int NXe = min(NX, n - u_lo), NSe = min(NS, n - (t0 - w));
            const int per_x = ((NXe + 31) >> 5) | 1, per_s = ((NSe + 31) >> 5) | 1;
            // 0. codes of residues u_lo-2 .. u_lo+NX-1 into shared memory (independent loads, issued together)
            for (int e0 = 0; e0 < NXe + 2; e0 += 32 * 12) {
                uint8_t cdv[12];
#pragma unroll
                for (int k = 0; k < 12; k++) {
                    const int e = e0 + 32 * k + lane;
                    const int u = u_lo - 2 + e;
                    cdv[k] = (e < NXe + 2 && u >= 0) ? src[u] : (uint8_t)0xff;
                }
#pragma unroll
                for (int k = 0; k < 12; k++) {
                    const int e = e0 + 32 * k + lane;
                    // outside the protein: pad; invalid input (> 21) is scored as X and reported by k_pack
                    if (e < NXe + 2) Cd[e] = cdv[k] == 0xff ? (uint8_t)kPad : (cdv[k] > 21 ? (uint8_t)0 : cdv[k]);
                }
            }
            __syncwarp();
            // 1. per-residue values (zero outside the protein: all tables are 0 for the pad code) and their prefix sums in
            // one go: lane l owns the run [l*per_x, l*per_x + per_x), adds its values up as it looks them up and stores the
            // running sums (same association as a scan of stored values: run sums, warp scan of the run totals, offsets)
            {
                const int lo = lane * per_x, hi = min(lo + per_x, NXe);
                double ra = 0, rb = 0, rc = 0;
                int rd = 0;
                for (int e = lo; e < hi; e++) {
                    const uint32_t cd = Cd[e + 2];
                    double pp = tab_p[cd];
                    // PAPA proline rule (:2652-2655): the second proline of PP / PxP is not scored
                    if (ks.adjust_prolines && cd == 13u && (Cd[e + 1] == 13 || Cd[e] == 13)) pp = 0.0;
                    ra = ra + tab_h[cd];
                    rb = rb + tab_l[cd];
                    rc = rc + pp;
                    rd = rd + ((int)((ks.charge_plus >> cd) & 1u) - (int)((ks.charge_minus >> cd) & 1u));
                    Xh[e] = ra;
                    Xl[e] = rb;
                    Xp[e] = rc;
                    Xc[e] = rd;
                }
                double ia = ra, ib = rb, ic = rc;
                int id = rd;
#pragma unroll
                for (int sft = 1; sft < 32; sft <<= 1) {
                    const double oa = __shfl_up_sync(0xffffffffu, ia, sft), ob = __shfl_up_sync(0xffffffffu, ib, sft);
                    const double oc = __shfl_up_sync(0xffffffffu, ic, sft);
                    const int od = __shfl_up_sync(0xffffffffu, id, sft);
                    if (lane >= sft) {
                        ia = ia + oa;
                        ib = ib + ob;
                        ic = ic + oc;
                        id = id + od;
                    }
                }
                const double ea = __shfl_up_sync(0xffffffffu, ia, 1), eb = __shfl_up_sync(0xffffffffu, ib, 1);
                const double ec = __shfl_up_sync(0xffffffffu, ic, 1);
                const int ed = __shfl_up_sync(0xffffffffu, id, 1);
                if (lane > 0) {
                    for (int e = lo; e < hi; e++) {
                        Xh[e] = Xh[e] + ea;
                        Xl[e] = Xl[e] + eb;
                        Xp[e] = Xp[e] + ec;
                        Xc[e] = Xc[e] + ed;
                    }
                }
                __syncwarp();
            }
            // 2. pass-1 window sums for centres t0-w .. t0+T+w-1 and the five pass-1 tracks.  S*[idx] replaces X*[idx]:
            // a window needs X*[idx+2w] (not yet overwritten: chunks ascend) and X*[idx-1], which is the own-position
            // value of the lane below (shuffle; lane 0 takes lane 31's value of the previous chunk).
            double ch_ = 0, cl_ = 0, cp_ = 0;
            int cc_ = 0;
            for (int i0 = 0; i0 < NSe; i0 += 32) {
                const int idx = i0 + lane;
                const bool in_rng = idx < NSe;
                const int pc = t0 - w + idx;
                const int eo = min(idx, NXe - 1);
                const double xoh = Xh[eo], xol = Xl[eo], xop = Xp[eo];
                const int xoc = Xc[eo];
                double lh = __shfl_up_sync(0xffffffffu, xoh, 1), ll = __shfl_up_sync(0xffffffffu, xol, 1);
                double lp = __shfl_up_sync(0xffffffffu, xop, 1);
                int lc = __shfl_up_sync(0xffffffffu, xoc, 1);
                if (lane == 0) {
                    lh = ch_;
                    ll = cl_;
                    lp = cp_;
                    lc = cc_;
                }
                ch_ = __shfl_sync(0xffffffffu, xoh, 31);
                cl_ = __shfl_sync(0xffffffffu, xol, 31);
                cp_ = __shfl_sync(0xffffffffu, xop, 31);
                cc_ = __shfl_sync(0xffffffffu, xoc, 31);
                double sh = 0, sl = 0, sp_ = 0;
                int scv = 0;
                if (in_rng && pc >= 0 && pc < n) {
                    const int ehi = min(pc + w, n - 1) - u_lo;  // beyond the protein everything is zero
                    const int elo = pc - w - 1 - u_lo;          // == idx - 1 >= -1
                    sh = Xh[ehi] - (elo >= 0 ? lh : 0.0);
                    sl = Xl[ehi] - (elo >= 0 ? ll : 0.0);
                    sp_ = Xp[ehi] - (elo >= 0 ? lp : 0.0);
                    scv = Xc[ehi] - (elo >= 0 ? lc : 0);
                    if (pc >= t0 && pc < t0 + kTrackTile) {
                        // one reciprocal per residue instead of four divisions (1 ulp, far inside the 1e-9 bar);
                        // interior windows have the full tap count and use the precomputed reciprocal
                        const int cnt = full - max(0, w - pc) - max(0, pc + w - (n - 1));
                        const double rc = cnt == full ? rfull : 1.0 / (double)cnt;
                        const double hyd = sh * rc;
                        const double chg = (double)scv * rc;
                        const double fi_p = (ks.cc0 * hyd + ks.cc1 * fabs(chg)) + ks.cc2;
                        g.out.hydro[ob + pc] = hyd;
                        g.out.charge[ob + pc] = chg;
                        g.out.fi[ob + pc] = fi_p;
                        g.out.plaac[ob + pc] = sl * rc;
                        g.out.papa[ob + pc] = sp_ * rc;
                        if (n == 1) {  // w clips to 0: the second pass returns the value itself (:2588-2589)
                            g.out.fix2[ob] = fi_p;
                            g.out.plaacx2[ob] = sl * rc;
                            g.out.papax2[ob] = sp_ * rc;
                        }
                    }
                }
                __syncwarp();  // every lane of the chunk has read its X* values
                if (in_rng) {
                    Sh[idx] = sh;
                    Sl[idx] = sl;
                    Sp[idx] = sp_;
                    Sc[idx] = abs(scv);
                }
            }
            __syncwarp();
            warp_scan4_inplace(Sh, Sl, Sp, Sc, NSe, per_s, lane);
            // 3. pass-2 tracks for centres t0 .. t0+T-1 (NaN outside [w, n-1-w], :2596-2601)
            if (n > 1) {
                for (int idx = lane; idx < kTrackTile; idx += 32) {
                    const int k = t0 + idx;
                    if (k >= n) break;
                    double f2 = nan(""), l2 = f2, p2 = f2;
                    if (k >= w && k <= n - 1 - w) {
                        const int ehi = idx + 2 * w;  // centre k+w in S* coordinates (S*[0] is centre t0-w)
                        const int elo = idx - 1;      // centre k-w-1
                        const double Th = Sh[ehi] - (elo >= 0 ? Sh[elo] : 0.0);
                        const double Tl = Sl[ehi] - (elo >= 0 ? Sl[elo] : 0.0);
                        const double Tp = Sp[ehi] - (elo >= 0 ? Sp[elo] : 0.0);
                        const int Tac = Sc[ehi] - (elo >= 0 ? Sc[elo] : 0);
                        const int ml = 2 * w - k, mr = 2 * w - (n - 1 - k);
                        const int Wi = Wfull - (ml > 0 ? (ml * (ml + 1)) >> 1 : 0) - (mr > 0 ? (mr * (mr + 1)) >> 1 : 0);
                        const double Wd = (double)Wi;
                        const double rW = Wi == Wfull ? rWfull : 1.0 / Wd;
                        f2 = ((ks.cc0 * Th + ks.cc1 * (double)Tac) + ks.cc2 * Wd) * rW;
                        l2 = Tl * rW;
                        p2 = Tp * rW;
                    }
                    g.out.fix2[ob + k] = f2;
                    g.out.plaacx2[ob + k] = l2;
                    g.out.papax2[ob + k] = p2;
                }
            }
            __syncwarp();
        }
    }
}

// ------------------------------------------------------------------------------------------------ host side
struct ResidueV2Plan {
    bool ok = false;           // false: parameters outside what these kernels support (fall back to residue_kernel.cuh)
    size_t fwd_smem = 0, bwd_smem = 0, trk_smem = 0;
    int nx = 0, per_x = 0, per_s = 0;
};

inline ResidueV2Plan residue_v2_plan(const KScalars& ks)
{
    ResidueV2Plan P;
    P.bwd_smem = kResFixedBytes;
    P.fwd_smem = kResFixedBytes;
    P.nx = kTrackTile + 4 * ks.w;
    const int ns = kTrackTile + 2 * ks.w;
    P.per_x = ((P.nx + 31) / 32) | 1;
    P.per_s = ((ns + 31) / 32) | 1;
    const size_t per_warp = ((size_t)P.nx * 28 + (size_t)P.nx + 64 + 15) & ~(size_t)15;
    P.trk_smem = per_warp * kTrackWarps;
    P.ok = P.trk_smem <= 200 * 1024 && P.fwd_smem <= 227 * 1024;
    return P;
}

// (the attribute belongs to the function, not to a ctx: raised once to the device's opt-in maximum, see plaac_create)
inline int residue_v2_setup(const ResidueV2Plan& P, int optin_bytes)
{
    if (!P.ok) return PLAAC_OK;
    if (raise_dynamic_smem_limit((const void*)k_res_bwd, optin_bytes, P.bwd_smem) != cudaSuccess) return PLAAC_E_CUDA;
    if (raise_dynamic_smem_limit((const void*)k_res_fwd, optin_bytes, P.fwd_smem) != cudaSuccess) return PLAAC_E_CUDA;
    if (raise_dynamic_smem_limit((const void*)k_res_tracks, optin_bytes, P.trk_smem) != cudaSuccess) return PLAAC_E_CUDA;
    return PLAAC_OK;
}

// Kernel order; aux streams (may be NULL) let the independent chains overlap:
//   st:   vit ------------\
//   aux3: tracks ---------+
//   aux1: bwd ------------+--> lpseq -> post -> bits   (on st)
//   aux2: fwd ------------/
// (the tracks only read the residue codes: beside the Viterbi pass instead of behind it)
// (Running the posterior chain on aux1 beside the tracks was measured slower: 6.2 vs 5.7 ms at 200 k proteins.)
inline int launch_residue_v2(const ResidueV2Plan& P, const ResArgs& ra, const TrackArgs& ta, int sm_count, cudaStream_t st,
                             cudaStream_t aux1, cudaStream_t aux2, cudaStream_t aux3, cudaEvent_t ev_fork, cudaEvent_t ev_j1,
                             cudaEvent_t ev_j2, cudaEvent_t ev_j3, int64_t* launches)
{
    const plaac_residue_out& out = ra.out;
    if (!out.post_bg || !out.post_prd || !out.charge || !out.hydro || !out.fi || !out.plaac || !out.papa || !out.fix2 ||
        !out.plaacx2 || !out.papax2)
        return PLAAC_E_INVALID;
    const int64_t nb = ra.bv.nbuckets;
    const bool fork = aux1 && aux2 && aux3;
    cudaStream_t s1 = fork ? aux1 : st, s2 = fork ? aux2 : st, s3 = fork ? aux3 : st;
    if (fork) {
        cudaEventRecord(ev_fork, st);
        cudaStreamWaitEvent(s1, ev_fork, 0);
        cudaStreamWaitEvent(s2, ev_fork, 0);
        cudaStreamWaitEvent(s3, ev_fork, 0);
    }
    // A small batch is bound by the dependent chain of its longest bucket: one warp alone on a scheduler partition takes
    // 240-280 cycles per residue step of the LUT recurrences, four warps on it 537 (scripts/gpu/micro/lse.cu).  With
    // 16 warps per CTA a yeast-sized set (188 buckets) crowded onto 12 SMs; the CTAs shrink until the buckets cover the SMs.
    int w_hmm = kResHmmThreads / 32, w_vit = kResThreads / 32;
    while (w_hmm > 1 && (nb + w_hmm - 1) / w_hmm < (int64_t)sm_count) w_hmm >>= 1;
    while (w_vit > 1 && (nb + w_vit - 1) / w_vit < (int64_t)sm_count) w_vit >>= 1;
    const unsigned g_vit = (unsigned)std::min<int64_t>((nb + w_vit - 1) / w_vit, (int64_t)sm_count * 8);
    const unsigned g_hmm = (unsigned)std::min<int64_t>((nb + w_hmm - 1) / w_hmm, (int64_t)sm_count * 2);
    const unsigned g_trk = (unsigned)std::min<int64_t>((ta.nprot + kTrackWarps - 1) / kTrackWarps, (int64_t)sm_count * 8);
    const unsigned g_bits = (unsigned)std::min<int64_t>(nb, (int64_t)sm_count * 8);
    const unsigned g_post = (unsigned)std::min<int64_t>((ra.bv.nslots + kResPostThreads / 32 - 1) / (kResPostThreads / 32) + 1, (int64_t)sm_count * 12);
    // The tracks join last on large batches: nothing behind them reads what they write, and the posterior / byte passes
    // then run beside their tail (200 k proteins: 5.53 -> 5.17 ms; a yeast-sized set loses 2 % to the extra sharing).
    const bool late = nb >= 1024;
    k_res_bwd<<<g_hmm, w_hmm * 32, P.bwd_smem, s1>>>(ra);
    k_res_fwd<<<g_hmm, w_hmm * 32, P.fwd_smem, s2>>>(ra);
    k_res_vit<<<g_vit, w_vit * 32, 0, st>>>(ra);
    k_res_tracks<<<g_trk, kTrackWarps * 32, P.trk_smem, s3>>>(ta);
    if (fork) {
        cudaEventRecord(ev_j1, s1);
        cudaEventRecord(ev_j2, s2);
        cudaEventRecord(ev_j3, s3);
        cudaStreamWaitEvent(st, ev_j1, 0);
        cudaStreamWaitEvent(st, ev_j2, 0);
        if (!late) cudaStreamWaitEvent(st, ev_j3, 0);
    }
    k_res_lpseq<<<(unsigned)((ra.bv.nprot + 255) / 256), 256, 0, st>>>(ra);
    k_res_post<<<g_post, kResPostThreads, 0, st>>>(ra);
    k_res_bits<<<g_bits, kResThreads, 0, st>>>(ra);
    if (fork && late) cudaStreamWaitEvent(st, ev_j3, 0);  // the tracks join last: nothing behind them reads what they write
    if (launches) *launches += 7;
    return cudaGetLastError() == cudaSuccess ? PLAAC_OK : PLAAC_E_CUDA;
}

}  // namespace plaac
