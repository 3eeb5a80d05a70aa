// Long-sequence path, summary mode (BASELINE config 5: titin-length and 100k-residue proteins).
//
// In the bucketed kernel one lane walks one protein, so a lone long protein costs its full dependent chain
// (~150 ns per residue: 15 ms for 100k residues).  Here a long protein's record is computed by four kernels:
//
//   k_long_post   (long_residue.cuh) one thread-block cluster per protein: the forward score, the Viterbi parse and
//                 the Viterbi score, bit for bit the jar's
//   k_long_score  TWO CTAs per protein (blockIdx.y), each with an ext copy of its own and one lane per chunk (<= 384
//                 chunks, 32 consecutive chunks per warp).  CTA 0, the sums and the searches:
//     sums        the plain sequential fp64 sums of plaac.java -- psum[] of the LLR window search (hss2 :1206-1257),
//                 hmm0's log-emission sum, the hydropathy mean.  Pass 1 sums every chunk in a chunk-local frame and a
//                 prefix over the chunk sums gives approximate absolute values.  That is exact mathematics but NOT the
//                 jar's rounding: at |s| ~ 3e5 every addition of the jar rounds to ulp = 5.8e-11 and the dropped low
//                 bits of the addends are the same at every step, so the jar's sums carry a systematic drift that a
//                 chunk-local frame does not have.  Pass 2 therefore re-runs every chunk in the jar's own binade,
//                 started from pass 1's absolute value: every addition has an operand of the running magnitude,
//                 rounding is monotone and commutes with shifts by multiples of the ulp, hence a chunk reproduces the
//                 jar's sequential values up to an EXACT shift.  Chunk increments and window differences are then
//                 exact multiples of the ulp and their ordered combination is the jar's number BIT FOR BIT.  The
//                 exception is an exact tie: round-half-even decides it by the parity of the sum, which a shift by an
//                 odd number of ulps changes.  The host lists the binades in which a table constant is such a tie
//                 (LongArgs::tie_mask); chunks there, and chunks in which the magnitude crosses a power of two (about
//                 one per binade), are redone sequentially from the exact values.  (k_long_post's recurrences get the
//                 same treatment; its forward recurrence has data-dependent addends and handles parity with two
//                 frames one ulp apart.)
//     searches    the LLR window maxima are merged in chunk order; the Q/N window and the charge sum are integer work.
//                 CTA 1, the windows (disorderreport :4866-5068): the running window sums restart 2w residues before
//                 the chunk; FoldIndex runs and the PAPA first-strict-maximum are reduced per chunk and merged in chunk
//                 order.
//   k_long_final  from k_long_post's parse: longestrun and the -1e6-masked CORE search with the exact binade jumps of
//                 k_core_search_jump, PrD expansion and PRDscore
//   k_long_fix    the two HMM scores, once k_long_post's scores and k_long_score's hmm0 sum are there
//
// Result: every column has the bits of the bucketed kernel, which has the bits of the jar.
#pragma once
#include "common.cuh"
#include "summary_kernel_v2.cuh"

namespace plaac {

constexpr int kLongThreads = 512;
constexpr int kLongChunkWarps = 12;
constexpr int kLongMaxChunks = kLongChunkWarps * 32;
constexpr int kLongMinChunk = 256;
constexpr int kLongPadTail = 128;  // ext bytes past the end are pad codes

// Chunk geometry of one long protein: C residues per chunk (a multiple of 32 that holds a whole CORE / MW window), K
// chunks (<= kLongMaxChunks).
__host__ __device__ inline void long_geometry(int64_t n, int c, int mw, int* C, int* K)
{
    int64_t cc = (n + kLongMaxChunks - 1) / kLongMaxChunks;
    cc = (cc + 31) & ~(int64_t)31;
    if (cc < kLongMinChunk) cc = kLongMinChunk;
    const int64_t wmin = (((c > mw ? c : mw) + 32) + 31) & ~(int64_t)31;
    if (cc < wmin) cc = wmin;
    *C = (int)cc;
    *K = (int)((n + cc - 1) / cc);
}
// Scratch bytes per array (one byte per residue and the pad tail) of one long protein; a multiple of 128.
__host__ __device__ inline int64_t long_scratch_need(int64_t n) { return (n + kLongPadTail + 127) & ~(int64_t)127; }

struct LongArgs {
    const uint8_t* codes;
    const int64_t* offsets;
    int64_t off_base;
    const int32_t* list;         // protein indices
    const int64_t* scratch_off;  // per listed protein, multiple of 128
    KScalars ks;
    const DeviceTables* tabs;
    plaac_summary* out;
    double* sum0_out;     // per listed protein: hmm0's log-emission sum, for k_long_fix
    uint8_t* ext;         // ext code per residue (same byte layout as the bucketed stream): CTA 0's copy
    uint8_t* ext_win;     // the same, CTA 1's copy
    uint32_t* vit;        // Viterbi bits, one word per 32 residues (k_long_final)
    int* errflag;
    // Round-half-even breaks the shift argument exactly at ties (an addend whose bits below the binade's ulp are
    // 1000...0): the rounding then depends on the parity of the sum.  The host lists the binades (bit b: values in
    // [2^b, 2^(b+1))) in which some table constant of a sum is such a tie; chunks there are redone sequentially.
    // [0] LLR psum (llr), [1] hmm0 sum (le0), [2] hydropathy sum.
    unsigned long long tie_mask[3];
};

struct LongShared {
    double le0[32];
    double llr[kTabN], hyd[kTabN], pap[kTabN], hydw[kTabN];
    // per chunk: windows (CTA 1)
    double p_tb[kLongMaxChunks], p_wb[kLongMaxChunks], p_vfi[kLongMaxChunks];
    int p_cen[kLongMaxChunks];
    int fi_pre[kLongMaxChunks], fi_suf[kLongMaxChunks], fi_sum[kLongMaxChunks], fi_max[kLongMaxChunks];
    unsigned char fi_all[kLongMaxChunks];
    // per chunk: sequential sums (psum[] of the LLR search, hmm0's emission sum, hydropathy sum): [0] LLR, [1] hmm0,
    // [2] hydropathy (CTA 0)
    double q_sum[3][kLongMaxChunks], q_min[3][kLongMaxChunks], q_max[3][kLongMaxChunks];  // pass 1, chunk-local
    double q_abs[3][kLongMaxChunks];                                                      // pass 1: value before the chunk
    double q_inc[3][kLongMaxChunks], q_mid[kLongMaxChunks], q_best[kLongMaxChunks];       // pass 2, exact
    int q_stop[kLongMaxChunks], m_best[kLongMaxChunks], m_stop[kLongMaxChunks], c_sum[kLongMaxChunks];
    unsigned char cross_q[3][kLongMaxChunks];
    // results of the combines
    double llr_best, sum0, sh;
    int llr_stop, csum, mw_best, mw_stop;
};

// Proteins of at least long_min residues are scored by the long-sequence path; the bucketed path sees them as empty.
__global__ void __launch_bounds__(256)
k_long_select(const int64_t* __restrict__ offsets, int64_t nprot, int64_t long_min,
              int32_t* __restrict__ list, int64_t* __restrict__ scratch_off,
              unsigned long long* __restrict__ counters /* [0] count, [1] scratch cursor, [2] count of >= big_min residues */,
              int64_t big_min)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nprot) return;
    const int64_t len = offsets[i + 1] - offsets[i];
    if (len < long_min) return;
    const unsigned long long slot = atomicAdd(&counters[0], 1ull);
    const unsigned long long need = (unsigned long long)long_scratch_need(len);
    list[slot] = (int32_t)i;
    scratch_off[slot] = (int64_t)atomicAdd(&counters[1], need);
    if (len >= big_min) atomicAdd(&counters[2], 1ull);
}

// barrier of the chunk warps only (the other warps leave after phase 0)
__device__ __forceinline__ void long_chunk_bar()
{
    // (barrier.sync without .aligned: the compiler may place the statement on both sides of a branch a warp has diverged
    // on -- compute-sanitizer's synccheck found warps arriving divergent at the aligned form; __syncwarp first)
    __syncwarp();
    asm volatile("barrier.sync 1, %0;" ::"n"(kLongChunkWarps * 32) : "memory");
}

// Automatic threshold: length bins from 1024 up (256-residue steps to 16384, then powers of two); the host picks the
// smallest bin edge that leaves at most one wave of long proteins (plaac_cuda.cu: choose_long_threshold).
constexpr int kLongBins = 78;
__host__ __device__ __forceinline__ int long_bin(int64_t len)
{
    if (len < 1024) return -1;
    if (len < 16384) return (int)((len - 1024) >> 8);
    int lg = 14;
    while (lg < 62 && (len >> (lg + 1)) != 0) lg++;
    const int b = 60 + (lg - 14);
    return b < kLongBins ? b : kLongBins - 1;
}
inline int64_t long_edge(int b) { return b < 60 ? 1024 + 256 * (int64_t)b : (int64_t)1 << (14 + b - 60); }

// per bin: [b] proteins, [kLongBins + b] scratch bytes, [2 * kLongBins + b] longest member
__global__ void __launch_bounds__(256)
k_long_levels(const int64_t* __restrict__ offsets, int64_t nprot, unsigned long long* __restrict__ bins)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nprot) return;
    const int64_t len = offsets[i + 1] - offsets[i];
    const int b = long_bin(len);
    if (b < 0) return;
    atomicAdd(&bins[b], 1ull);
    atomicAdd(&bins[kLongBins + b], (unsigned long long)long_scratch_need(len));
    atomicMax(&bins[2 * kLongBins + b], (unsigned long long)len);
}

// Grid (long proteins, 2): blockIdx.y = 0 computes the sums, the MW and LLR searches and the means; 1 the window
// columns (FoldIndex runs, PAPA centre and its values).
__global__ void __launch_bounds__(kLongThreads, 1) k_long_score(LongArgs g)
{
    extern __shared__ __align__(16) unsigned char long_smem[];
    LongShared& sm = *reinterpret_cast<LongShared*>(long_smem);
    const KScalars& ks = g.ks;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int32_t prot = g.list[blockIdx.x];
    const int64_t so = g.scratch_off[blockIdx.x];
    const int n = (int)(g.offsets[prot + 1] - g.offsets[prot]);
    const uint8_t* src = g.codes + (g.offsets[prot] - g.off_base);
    const bool win = blockIdx.y == 1;
    uint8_t* __restrict__ ext = (win ? g.ext_win : g.ext) + so;
    const int c = ks.core_len, w = ks.w, mw = ks.mw_window;
    int C, K;
    long_geometry(n, c, mw, &C, &K);

    // ---- tables
    {
        const DeviceTables* T = g.tabs;
        if (tid < 32) sm.le0[tid] = T->le0[tid];
        if (tid < kTabN) {
            sm.llr[tid] = T->llr[tid];
            sm.hyd[tid] = T->hyd[tid];
            sm.hydw[tid] = T->hydw[tid];
            sm.pap[tid] = T->pap[tid];
        }
    }
    // ---- phase 0: ext codes (k_pack's byte layout: code | PAPA proline mask << 5 | charge class << 6)
    {
        int bad = 0;
        // eight residues per thread and trip, all loads issued before the first use (a single byte load per trip left
        // the CTA waiting on DRAM latency: 0.1 ms of the 1.4 ms at 100 k residues)
        constexpr int kU = 8;
        for (int base = 0; base < n; base += kLongThreads * kU) {
            uint32_t cd[kU], p1[kU], p2[kU];
#pragma unroll
            for (int u = 0; u < kU; u++) {
                const int i = base + u * kLongThreads + tid;
                cd[u] = i < n ? (uint32_t)src[i] : 0u;
                p1[u] = (i < n && i >= 1) ? (uint32_t)src[i - 1] : 0u;
                p2[u] = (i < n && i >= 2) ? (uint32_t)src[i - 2] : 0u;
            }
#pragma unroll
            for (int u = 0; u < kU; u++) {
                const int i = base + u * kLongThreads + tid;
                if (i >= n) continue;
                uint32_t c0 = cd[u];
                if (c0 > 21u) {
                    bad = 1;
                    c0 = 0;
                }
                uint32_t e = c0;
                if (ks.adjust_prolines && c0 == 13u && (p1[u] == 13u || p2[u] == 13u)) e |= (uint32_t)kPapaMaskBit;
                if ((ks.charge_plus >> c0) & 1u)
                    e |= 0x40u;
                else if ((ks.charge_minus >> c0) & 1u)
                    e |= 0xc0u;
                ext[i] = (uint8_t)e;
            }
        }
        for (int i = n + tid; i < n + kLongPadTail; i += kLongThreads) ext[i] = (uint8_t)kPad;
        if (bad) atomicOr(g.errflag, 1);
    }
    __syncthreads();
    if (wid >= kLongChunkWarps) return;

    const int k = tid;
    const bool live = k < K;
    const int cs = k * C, ce = min(n, cs + C);
    // ================= pass 1: chunk-local frame =================
    if (live && !win) {
        // the chunk-local sums of the three sequential-sum columns (running extremes for the binade test), the charge
        // sum and the Q/N window: independent dependency chains in one loop
        double q0 = 0, q1 = 0, q2 = 0, mn0 = 0, mn1 = 0, mn2 = 0, mx0 = 0, mx1 = 0, mx2 = 0;
        int cq = 0;
        int qn = 0, mbest = -1, mstop = -1;
        for (int t = max(0, cs - mw); t < cs; t++) qn += (int)((ks.qn_mask >> (ext[t] & 31)) & 1u);
        auto stats = [&](int t, uint32_t e) {
            q0 = q0 + sm.llr[e & 31];
            q1 = q1 + sm.le0[e & 31];
            q2 = q2 + sm.hyd[e & 63];
            mn0 = fmin(mn0, q0), mx0 = fmax(mx0, q0);
            mn1 = fmin(mn1, q1), mx1 = fmax(mx1, q1);
            mn2 = fmin(mn2, q2), mx2 = fmax(mx2, q2);
            cq += (int)(int8_t)e >> 6;
            // Q/N window :764-771: first strict maximum of the count in [t-mw+1, t] (n >= mw here)
            qn += (int)((ks.qn_mask >> (e & 31)) & 1u);
            if (t >= mw) qn -= (int)((ks.qn_mask >> (ext[t - mw] & 31)) & 1u);
            if (t >= mw - 1 && qn > mbest) {
                mbest = qn;
                mstop = t;
            }
        };
        int t0 = cs;
        if (k == 0) {
            stats(0, ext[0]);
            t0 = 1;
        }
#pragma unroll 4
        for (int t = t0; t < ce; t++) stats(t, ext[t]);
        sm.q_sum[0][k] = q0, sm.q_min[0][k] = mn0, sm.q_max[0][k] = mx0;
        sm.q_sum[1][k] = q1, sm.q_min[1][k] = mn1, sm.q_max[1][k] = mx1;
        sm.q_sum[2][k] = q2, sm.q_min[2][k] = mn2, sm.q_max[2][k] = mx2;
        sm.c_sum[k] = cq;
        sm.m_best[k] = mbest;
        sm.m_stop[k] = mstop;
    }
    if (live && win) {
        // ---- sliding windows: FoldIndex runs and the PAPA centre over the positions this chunk owns
        const int off1 = 2 * w + 1, off2 = 4 * w + 2;
        const int full = 2 * w + 1, Wfull = full * full;
        const int t_start = max(0, cs - 2 * w);
        const int t_last = min(ce + 2 * w, n + w) - 1;
        int halfw = ks.h_fi;
        if (halfw > n / 2) halfw = n / 2;
        const int fi_hi = n - halfw, edge_hi = n - 1 - w;
        double SLh = 0, SGh = 0, Th = 0, Dp = 0, Tp = 0;
        int SLc = 0, SGc = 0, Tac = 0;
        double Tb = 0, Wb = 1, vfib = 0;
        int pcen = -1;
        int cur = 0, pre = 0, insum = 0, inmax = 0;
        bool all = true;
#pragma unroll 8
        for (int t = t_start; t <= t_last; t++) {
            const uint32_t e0 = (t < n) ? ext[t] : (uint32_t)kPad;
            const uint32_t e1 = (t - off1 >= t_start) ? ext[t - off1] : (uint32_t)kPad;
            const uint32_t e2 = (t - off2 >= t_start) ? ext[t - off2] : (uint32_t)kPad;
            const double hy0 = sm.hydw[e0 & 63], hy1 = sm.hydw[e1 & 63], hy2 = sm.hydw[e2 & 63];
            const double pa0 = sm.pap[e0 & 63], pa1 = sm.pap[e1 & 63], pa2 = sm.pap[e2 & 63];
            const int ch0 = (int)(int8_t)e0 >> 6, ch1 = (int)(int8_t)e1 >> 6, ch2 = (int)(int8_t)e2 >> 6;
            SLh = (SLh + hy0) - hy1;
            SGh = (SGh + hy1) - hy2;
            Th = (Th + SLh) - SGh;
            Dp = Dp + ((pa0 + pa2) - (pa1 + pa1));
            Tp = Tp + Dp;
            SLc += ch0 - ch1;
            SGc += ch1 - ch2;
            const int aSL = abs(SLc);
            Tac += aSL - abs(SGc);
            const int p = t - w;
            if (p >= cs && p < ce && p >= halfw && p < fi_hi) {
                const double c2 = ks.cc2 * (double)(full - max(0, w - p) - max(0, p - edge_hi));
                const double fis = (ks.cc0 * SLh + ks.cc1 * (double)aSL) + c2;
                if (fis < 0) {
                    cur += 1;
                    if (p == halfw) cur += halfw;           // a run from the first scanned position snaps to 0
                    if (p == fi_hi - 1) cur += n - 1 - p;   // one reaching the last scanned position snaps to n-1
                } else {
                    if (all) {
                        pre = cur;
                        all = false;
                    } else if (cur >= 5) {
                        insum += cur;
                        inmax = max(inmax, cur);
                    }
                    cur = 0;
                }
            }
            const int kk = p - w;
            if (kk >= cs && kk < ce && kk >= w && kk <= edge_hi) {
                const int ml = 2 * w - kk, mr = kk - (edge_hi - w);
                const double Wd =
                    (double)(Wfull - (ml > 0 ? (ml * (ml + 1)) >> 1 : 0) - (mr > 0 ? (mr * (mr + 1)) >> 1 : 0));
                const double vfi = (ks.cc0 * Th + ks.cc1 * (double)Tac) + ks.cc2 * Wd;
                if ((pcen < 0 || Tp * Wb > Tb * Wd) && vfi < 0) {
                    Tb = Tp;
                    Wb = Wd;
                    vfib = vfi;
                    pcen = kk;
                }
            }
        }
        sm.fi_all[k] = all ? 1 : 0;
        sm.fi_pre[k] = all ? cur : pre;
        sm.fi_suf[k] = cur;
        sm.fi_sum[k] = insum;
        sm.fi_max[k] = inmax;
        sm.p_cen[k] = pcen;
        sm.p_tb[k] = Tb;
        sm.p_wb[k] = Wb;
        sm.p_vfi[k] = vfib;
    }
    long_chunk_bar();

    if (win) {
        if (tid != 0) return;
        // FoldIndex runs (:5010-5059) and PAPA centre (:4941-4948) merged in chunk order
        int open = 0, num = 0, mx = 0;
        int pcen = -1;
        double Tb = 0, Wb = 1, vfib = 0;
        for (int kk = 0; kk < K; kk++) {
            if (sm.fi_all[kk])
                open += sm.fi_pre[kk];
            else {
                const int r = open + sm.fi_pre[kk];
                if (r >= 5) {
                    num += r;
                    mx = max(mx, r);
                }
                num += sm.fi_sum[kk];
                mx = max(mx, sm.fi_max[kk]);
                open = sm.fi_suf[kk];
            }
            if (sm.p_cen[kk] >= 0 && (pcen < 0 || sm.p_tb[kk] * Wb > Tb * sm.p_wb[kk])) {
                Tb = sm.p_tb[kk];
                Wb = sm.p_wb[kk];
                vfib = sm.p_vfi[kk];
                pcen = sm.p_cen[kk];
            }
        }
        if (open >= 5) {
            num += open;
            mx = max(mx, open);
        }
        plaac_summary* r = g.out + prot;
        r->fi_numaa = num;
        r->fi_maxrun = mx;
        r->papa_center = pcen;
        if (pcen >= 0) {
            const double prop = Tb / Wb;
            r->papa_combo = prop;
            r->papa_prop = prop;
            r->papa_fi = vfib / Wb;
            const int full = 2 * w + 1;
            const int q0 = max(pcen - 2 * w, 0), q1 = min(pcen + 2 * w, n - 1);
            double sc = 0.0, den = 0.0, t2 = 0.0;
            for (int q = q0; q <= q1; q++) {
                const double x = sm.llr[ext[q] & 63];
                const int dist = abs(q - pcen);
                if (dist <= w) {
                    den = den + 1.0;
                    sc = sc + 1.0 * x;
                }
                t2 = t2 + x * (double)(full - dist);
            }
            r->papa_llr = sc / den;
            r->papa_llr2 = t2 / Wb;
        } else {
            r->papa_combo = -INFINITY;
            r->papa_prop = r->papa_fi = r->papa_llr = r->papa_llr2 = nan("");
        }
        return;
    }

    // ================= combine 1: approximate absolute values (they only fix the binade of pass 2) =================
    if (wid == 0 && lane < 3) {
        double run = 0.0;
        for (int kk = 0; kk < K; kk++) {
            sm.q_abs[lane][kk] = run;
            run += sm.q_sum[lane][kk];
        }
    }
    long_chunk_bar();
    // ================= pass 2: the jar's own binade =================
    // Every fp64 addition of a sum has one operand of the running magnitude, so it rounds to a multiple of that
    // magnitude's ulp; rounding is monotone and commutes with shifts by multiples of the ulp as long as no operand changes
    // its binade.  Re-run from an approximate absolute value, a chunk therefore reproduces the jar's sequential values up
    // to an EXACT shift: increments and window differences are exact multiples of the ulp and their ordered combination
    // is the jar's number bit for bit.  Chunks in which the magnitude crosses a power of two (about one per binade) are
    // redone sequentially from the exact values.
    if (live && k >= 1) {
        double lagsum = 0;
        for (int t = cs - c; t < cs; t++) lagsum += sm.llr[ext[t] & 31];
        double lag = sm.q_abs[0][k] - lagsum;  // approximate psum before residue cs-c: fixes the frame
        double lead = lag;
        for (int t = cs - c; t < cs; t++) lead = lead + sm.llr[ext[t] & 31];
        const double lead0 = lead;
        double best = -INFINITY, mid = lead;
        int stop = -1;
        const double x10 = sm.q_abs[1][k], x20 = sm.q_abs[2][k];
        double x1 = x10, x2 = x20;
#pragma unroll 4
        for (int t = cs; t < ce; t++) {
            const uint32_t e = ext[t];
            lead = lead + sm.llr[e & 31];
            lag = lag + sm.llr[ext[t - c] & 31];
            const double d = lead - lag;  // exact, and the jar's number
            if (d > best) {
                best = d;
                stop = t;
            }
            if (t == ce - c - 1) mid = lead;
            x1 = x1 + sm.le0[e & 31];
            x2 = x2 + sm.hyd[e & 63];
        }
        sm.q_inc[0][k] = lead - lead0;
        sm.q_mid[k] = mid - lead0;
        sm.q_best[k] = best;
        sm.q_stop[k] = stop;
        sm.q_inc[1][k] = x1 - x10;
        sm.q_inc[2][k] = x2 - x20;
    }
    if (live) {
        // crossing test over every value the running sum takes in the region (for the LLR search the lagged sum
        // starts c residues before the chunk, i.e. inside the previous chunk)
#pragma unroll
        for (int q = 0; q < 3; q++) {
            double mn = sm.q_abs[q][k] + sm.q_min[q][k], mx = sm.q_abs[q][k] + sm.q_max[q][k];
            if (q == 0 && k >= 1) {
                mn = fmin(mn, sm.q_abs[0][k - 1] + sm.q_min[0][k - 1]);
                mx = fmax(mx, sm.q_abs[0][k - 1] + sm.q_max[0][k - 1]);
            }
            const double lo = fmin(fabs(mn), fabs(mx)) * (1.0 - 1e-6), hi = fmax(fabs(mn), fabs(mx)) * (1.0 + 1e-6);
            const bool cross = k == 0 || !(mn > 0.0 || mx < 0.0) || !(lo >= 1.0) ||
                               (__double2hiint(lo) >> 20) != (__double2hiint(hi) >> 20) ||
                               ((g.tie_mask[q] >> (((__double2hiint(lo) >> 20) & 0x7ff) - 1023)) & 1ull);
            sm.cross_q[q][k] = cross ? 1 : 0;
        }
        if (k == 0) {
            // first chunk: the true chains from residue 0 (hss2 :1206-1257, mean() :1584, hmm0's emission sum)
            double ps = 0, psl = 0, best = 0, mid = 0;
            int stop = -2;
            double s0 = 0, shy = 0;
#pragma unroll 8
            for (int t = 0; t < ce; t++) {
                const uint32_t e = ext[t];
                ps = ps + sm.llr[e & 31];
                if (t >= c) psl = psl + sm.llr[ext[t - c] & 31];
                if (t >= c - 1) {
                    const double d = ps - psl;
                    if (t == c - 1 || d > best) {
                        best = d;
                        stop = t;
                    }
                }
                if (t == ce - c - 1) mid = ps;
                s0 = (t == 0) ? sm.le0[e & 31] : s0 + sm.le0[e & 31];
                shy = shy + sm.hyd[e & 63];
            }
            sm.q_inc[0][0] = ps, sm.q_mid[0] = mid, sm.q_best[0] = best, sm.q_stop[0] = stop;
            sm.q_inc[1][0] = s0;
            sm.q_inc[2][0] = shy;
        }
    }
    long_chunk_bar();
    // ================= combine 2: exact, in chunk order =================
    if (wid == 0 && lane == 0) {
        // LLR window search: chunk maxima in order (first strict maximum), crossing chunks redone from exact values
        double P = sm.q_inc[0][0], Pl = sm.q_mid[0];
        double best = sm.q_best[0];
        int stop = sm.q_stop[0];
        for (int kk = 1; kk < K; kk++) {
            const int s = kk * C, e = min(n, s + C);
            double cand, Pl_next = P;
            int cstop;
            if (!sm.cross_q[0][kk]) {
                cand = sm.q_best[kk];
                cstop = sm.q_stop[kk];
                Pl_next = P + sm.q_mid[kk];
                P = P + sm.q_inc[0][kk];
            } else {
                double lead = P, lag = Pl;
                cand = -INFINITY;
                cstop = -1;
#pragma unroll 8
                for (int t = s; t < e; t++) {
                    lead = lead + sm.llr[ext[t] & 31];
                    lag = lag + sm.llr[ext[t - c] & 31];
                    const double d = lead - lag;
                    if (d > cand) {
                        cand = d;
                        cstop = t;
                    }
                    if (t == e - c - 1) Pl_next = lead;
                }
                P = lead;
            }
            if (cand > best) {
                best = cand;
                stop = cstop;
            }
            Pl = Pl_next;
        }
        sm.llr_best = best;
        sm.llr_stop = stop;
    } else if (wid == 1 && lane < 2) {
        // hmm0's emission sum (lane 0) and the hydropathy sum (lane 1)
        const int q = 1 + lane;
        double x = sm.q_inc[q][0];
        for (int kk = 1; kk < K; kk++) {
            if (!sm.cross_q[q][kk])
                x = x + sm.q_inc[q][kk];
            else {
                const int s = kk * C, e = min(n, s + C);
                if (q == 1)
                    for (int t = s; t < e; t++) x = x + sm.le0[ext[t] & 31];
                else
                    for (int t = s; t < e; t++) x = x + sm.hyd[ext[t] & 63];
            }
        }
        if (q == 1)
            sm.sum0 = x;
        else
            sm.sh = x;
    } else if (wid == 2 && lane == 0) {
        int best = sm.m_best[0], stop = sm.m_stop[0], cq = sm.c_sum[0];
        for (int kk = 1; kk < K; kk++) {
            if (sm.m_best[kk] > best) {
                best = sm.m_best[kk];
                stop = sm.m_stop[kk];
            }
            cq += sm.c_sum[kk];
        }
        sm.mw_best = best;
        sm.mw_stop = stop;
        sm.csum = cq;
    }
    long_chunk_bar();

    if (tid != 0) return;
    plaac_summary* r = g.out + prot;
    r->prot_len = n;
    r->mw_score = sm.mw_best;
    r->mw_start = sm.mw_stop - mw + 1;
    r->mw_end = sm.mw_stop;
    r->llr = sm.llr_best;
    r->llr_start = sm.llr_stop - c + 1;
    r->llr_end = sm.llr_stop;
    const double mh = (1.0 * sm.sh) / (double)n;
    const double mc = (1.0 * (double)sm.csum) / (double)n;
    r->fi_meanhydro = mh;
    r->fi_meancharge = mc;
    r->fi_meancombo = (ks.cc2 + ks.cc1 * fabs(mc)) + ks.cc0 * mh;
    g.sum0_out[blockIdx.x] = sm.sum0;
}

// The Viterbi-dependent columns of a long protein, from k_long_post's parse: Viterbi bytes -> bit words, longestrun
// (:1787-1804), the -1e6-masked CORE search with PrD expansion and PRDscore (:816-873), in reference order; masked
// stretches are applied as exact binade jumps when the masking constant is a negative integer.  It needs nothing from
// k_long_score (residue codes straight from the input), so it runs behind k_long_post while k_long_score is still at
// work; k_long_fix then writes the two HMM scores.
constexpr int kLongFinalThreads = 256;
__global__ void __launch_bounds__(kLongFinalThreads)
k_long_final(LongArgs g, const uint8_t* __restrict__ vbytes_all, const uint8_t* __restrict__ vit_out, int64_t res_base)
{
    __shared__ double llr_s[kTabN];
    __shared__ int s_all[kLongFinalThreads], s_pre[kLongFinalThreads], s_suf[kLongFinalThreads], s_max[kLongFinalThreads];
    __shared__ unsigned char s_any[kLongFinalThreads];  // the thread's range of words holds a Viterbi-1 residue
    const int tid = threadIdx.x;
    const int32_t prot = g.list[blockIdx.x];
    const int64_t so = g.scratch_off[blockIdx.x];
    const int n = (int)(g.offsets[prot + 1] - g.offsets[prot]);
    const uint8_t* __restrict__ src = g.codes + (g.offsets[prot] - g.off_base);
    // the parse lies in the caller's per-residue array if there is one, else in scratch
    const uint8_t* __restrict__ vb = vit_out ? vit_out + (g.offsets[prot] - res_base) : vbytes_all + so;
    uint32_t* __restrict__ vit = g.vit + (so >> 5);
    const KScalars& ks = g.ks;
    const int c = ks.core_len;
    if (tid < kTabN) llr_s[tid] = g.tabs->llr[tid];
    // ---- bytes -> bit words; per-thread run statistics of a contiguous range of words
    const int nwords = (n + 31) >> 5;
    const int per = (nwords + kLongFinalThreads - 1) / kLongFinalThreads;
    {
        const int w_lo = tid * per, w_hi = min(nwords, w_lo + per);
        int cur = 0, pre = 0, inmax = 0;
        bool closed = false;
        uint32_t any = 0;
        for (int j = w_lo; j < w_hi; j++) {
            uint32_t word = 0;
            const int t_hi = min(n, 32 * j + 32);
            for (int t = 32 * j; t < t_hi; t++) {
                const uint32_t v = vb[t] & 1u;
                word |= v << (t & 31);
                if (v)
                    cur++;
                else {
                    if (!closed) {
                        pre = cur;
                        closed = true;
                    } else
                        inmax = max(inmax, cur);
                    cur = 0;
                }
            }
            vit[j] = word;
            any |= word;
        }
        s_any[tid] = any ? 1 : 0;
        s_all[tid] = closed ? 0 : 1;      // the range is one run of ones (or empty)
        s_pre[tid] = closed ? pre : cur;  // ones at its start
        s_suf[tid] = cur;                 // ones at its end
        s_max[tid] = inmax;
    }
    __syncthreads();
    if (tid != 0) return;
    plaac_summary* r = g.out + prot;
    auto code = [&](int p) -> uint32_t {
        const uint32_t cd = src[p];
        return cd > 21u ? 0u : cd;
    };
    int open = 0, mx = 0;
    for (int k = 0; k < kLongFinalThreads; k++) {
        if (s_all[k])
            open += s_pre[k];
        else {
            mx = max(mx, max(open + s_pre[k], s_max[k]));
            open = s_suf[k];
        }
    }
    mx = max(mx, open);
    r->vit_maxrun = mx;
    r->core_start = -1;
    r->core_end = -2;
    r->prd_start = -1;
    r->prd_end = -2;
    r->core_score = nan("");
    r->prd_score = 0.0;
    if (mx < c) return;
    const double big_neg = ks.big_neg;
    const bool can_jump = big_neg < 0 && big_neg == floor(big_neg) && big_neg >= -4194304.0;
    double ps = 0.0, lag = 0.0, best = -INFINITY, runsum = 0.0, prd_sc = 0.0;
    int bstop = -1, run = 0, last = 0, run_start = 0, prd_s = -1, prd_e = -2;
    bool hit = false;
    for (int j = 0; j < nwords; j++) {
        if (j % per == 0 && !s_any[j / per]) {  // a range without a Viterbi-1 residue is one masked stretch
            j += per - 1;
            continue;
        }
        uint32_t bits = vit[j];
        while (bits) {
            const int i = __ffs((int)bits) - 1;
            bits &= bits - 1;
            const int p = 32 * j + i;
            if (p != last) {
                if (hit) {
                    prd_s = run_start;
                    prd_e = last - 1;
                    prd_sc = runsum;
                    hit = false;
                }
                if (can_jump)
                    ps = masked_jump(ps, p - last, big_neg);
                else
                    for (int q = last; q < p; q++) ps = ps + big_neg;
                run = 0;
            }
            if (run == 0) {
                lag = ps;
                run_start = p;
                runsum = 0.0;
            }
            const double x = llr_s[code(p)];
            ps = ps + x;
            runsum = runsum + x;
            if (run >= c - 1) {
                const double d = ps - lag;
                if (d > best) {
                    best = d;
                    bstop = p;
                    hit = true;
                }
                lag = lag + llr_s[code(p - c + 1)];
            }
            run++;
            last = p + 1;
        }
    }
    if (hit) {
        prd_s = run_start;
        prd_e = last - 1;
        prd_sc = runsum;
    }
    if (best > big_neg / 2) {
        r->core_start = bstop - c + 1;
        r->core_end = bstop;
        r->core_score = best;
        r->prd_start = prd_s;
        r->prd_end = prd_e;
        r->prd_score = prd_sc;
    }
}

// HMMall = lmarginalprob - sum0, HMMvit = lviterbiprob - sum0 (:790-800) once k_long_post (scores) and k_long_score (sum0) are done
__global__ void __launch_bounds__(128) k_long_fix(LongArgs g, const double* __restrict__ hmm_out, int nlong)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nlong) return;
    plaac_summary* r = g.out + g.list[i];
    const double sum0 = g.sum0_out[i];
    r->hmm_all = hmm_out[2 * i] - sum0;
    r->hmm_vit = hmm_out[2 * i + 1] - sum0;
}

}  // namespace plaac
