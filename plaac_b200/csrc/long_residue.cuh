// Long-sequence path on a thread-block cluster: the per-residue arrays of proteins the bucketed kernels would walk in a
// single lane (plotsomefastas :610-647 on titin-length proteins: posteriorl :3349-3411, mapdecodel :4032-4045,
// viterbidecodel :3077-3121) and, in records-only mode, the HMM columns of their summary record (forward score, Viterbi
// parse and score; the other columns: long_kernel.cuh).
//
// ONE THREAD-BLOCK CLUSTER per long protein (1 or 8 CTAs x 512 lanes), one lane per chunk of >= 32 residues.  Forward and
// backward LUT recurrences both get the binade-frame treatment of long_kernel.cuh, the Viterbi recurrence its max-plus
// transfer matrices:
//
//   pass 1   chunk-local frame: forward / backward after a 256-residue warm-up, the chunk's 2x2 max-plus matrix; prefix /
//            suffix sums and a Kogge-Stone matrix scan over warp shuffles give approximate absolute values at every chunk
//            boundary (they only decide binades); the CTA totals cross the cluster through DISTRIBUTED SHARED MEMORY
//   pass 2   the jar's own binade: two frames one ulp apart from pass 1's d (64-residue warm-up), two exact Viterbi frames
//   carry    one lane per chain walks the chunks in order and accepts the frame that enters the chunk an even number of
//            ulps from the exact value with exactly the bits of d = x1 - x0 the previous chunk left with (else it redoes the
//            chunk sequentially: binade crossings, |x| < 1024, uncoalesced warm-ups); chunks known beforehand to be linked
//            cost one addition.  The exact state at every chunk boundary is kept.  Across the CTAs the walk is a relay:
//            the walker writes its exact state into the next CTA's shared memory (DSMEM), fences at cluster scope and sets
//            a flag the next walker polls with back-off (forward and Viterbi: rank r -> r+1, backward: r -> r-1)
//   pass 3   every lane re-runs its chunk from the EXACT boundary state: backward first (b into scratch), then forward,
//            which leaves a + b per state in scratch -- the jar's a[][] and b[][] bit for bit; Viterbi chunks are traced
//            back in parallel from the end states (a warp-parallel suffix composition of the chunks' choice maps)
//   pass 4   all threads, coalesced: pp = exp((a + b) - lpseq) (:3401-3405), MAP byte = pp1 > pp0
//
// Small chunks make the sequential part cheap: a binade crossing costs its 2-3 chunks of 32-200 residues instead of a
// 288-residue chunk, and chunks whose warm-up reaches the protein's start (end) run the true chain and are exact as they are.
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"
#include "long_kernel.cuh"
#include "summary_kernel_v2.cuh"

namespace plaac {
namespace cg = cooperative_groups;

constexpr int kLpThreads = 512;   // chunk lanes per CTA
constexpr int kLpMinChunk = 32;
constexpr int kLpWarm2 = 64;      // warm-up residues of pass 2, which starts from pass 1's d (within a few ulps of the jar's)
constexpr int kLpBigCluster = 8;  // CTAs per protein of at least kLpBigMin residues
constexpr int kLpBigMin = 32768;  // (an edge of k_long_levels' length bins: the host counts the classes from them)
// Boundary scratch: five planes (gA, gB, gV0, gV1, bytes) of bnd_plane doubles; a protein's row starts at scratch_off / 32
// in every plane and has (n + 128) / 32 >= K + 2 entries (K <= n / 32 + 1 chunks), so the scratch is 1.25 bytes per long residue
// however many long proteins there are.
constexpr int kLpBndPlanes = 5;

struct LongPostArgs {
    const uint8_t* codes;
    const int64_t* offsets;
    int64_t off_base;            // codes[offsets[p] - off_base] is residue 0 of protein p
    int64_t res_base;            // out.*[offsets[p] - res_base] likewise
    const int32_t* list;         // k_long_select's list
    const int64_t* scratch_off;  // ... and scratch cursor (>= n + 128 per protein, multiple of 128)
    KScalars ks;
    const DeviceTables* tabs;
    plaac_residue_out out;
    double* S0;                  // scratch planes, indexed scratch_off + t: b0 then a0 + b0
    double* S1;
    double* bnd;                 // kLpBndPlanes planes of bnd_plane doubles: approximate a0 / b0 / Viterbi scores at the chunk boundaries
    int64_t bnd_plane;
    double* lpseq;               // per listed protein
    int warm;                    // warm-up residues of pass 1 (rounded up to whole chunks): d coalesces from a generic start
    int cluster;                 // CTAs per protein of this launch; the launch handles proteins of its size class only
    int64_t big_min;             // class boundary: n >= big_min belongs to the kLpBigCluster launch
    unsigned long long* redone;  // statistics: chunks redone sequentially although they had frames
    // Viterbi parse (viterbidecodel :3077-3121), for records and for out.vit: chunk transfer matrices, a max-plus scan
    // for the binades, two exact frames per chunk, exact combine, parallel traceback
    int want_vit;
    int want_post;               // 0: records only (summary mode): forward + Viterbi, no backward pass, no per-residue arrays
    double* hmm_out;             // per listed protein {lmarginalprob, lviterbiprob} (:3369-3375, :3102-3108) for k_long_final
    uint8_t* vbytes;             // Viterbi parse, one byte per residue at scratch_off + t, when out.vit is NULL
    uint8_t* tb;                 // 4 traceback bits per residue, indexed scratch_off + t
    unsigned long long vit_tie_mask;  // binades in which a Viterbi constant is an exact rounding tie (plaac_create)
    int* errflag;                // invalid residue codes (> 21) are scored as X and reported, as by k_pack
};

struct LpShared {
    double2 lut2[PLAAC_LUT_LEN + 1];
    double2 le[32];
    // pass 1: chunk increments and their local scans
    double inc[2][kLpThreads];
    // pass 2 per direction (0 forward, 1 backward): two frames
    double g_inc[2][2][kLpThreads], g_ea0[2][2][kLpThreads], g_den[2][2][kLpThreads], g_dex[2][2][kLpThreads];
    // exact state at the chunk's entry (forward: at cs-1, backward: at ce), filled by the carry walk
    double ent0[2][kLpThreads], ent1[2][kLpThreads];
    unsigned char mode[2][kLpThreads];  // 0 frames, 1 no frames (redo), 2 true chain (g_ea0/g_den[.][0] = exact entry, [.][1] = exact exit)
    // typ: both frames agree (same d at entry, same increment, same d at exit, entries an odd number of ulps apart), so
    // the chunk is accepted iff the exact d it is entered with has the bits of its frames' d.  link: typ, the chunk
    // before it in walking order is typ too and leaves with exactly that d -- known without the exact values.
    unsigned char typ[2][kLpThreads], link[2][kLpThreads];
    double tot[2];                      // pass 1: this CTA's total increment per direction
    double carry[2][2];                 // relay: exact state handed over by the neighbour CTA
    int carry_acc[2];                   // ... and whether its last chunk was accepted with its frames
    // Viterbi: chunk transfer matrix [.][0] 0->0, [1] 0->1, [2] 1->0, [3] 1->1 (pass 1: chunk-local, then its scan; pass 2: exact
    // frame, relative to its entry score)
    alignas(16) double vMi[kLpThreads][4];
    double vtot[4], vcarry[2];  // (interleaved: the walker loads a chunk's four entries with two 128-bit loads)
    unsigned char vcross[kLpThreads], vchoice[kLpThreads], vend[kLpThreads];
    double vE0, vE1;                    // exact scores at the first chunk's last residue
    unsigned char vall[kLpBigCluster * kLpThreads + 8];  // the cluster's choice bytes, staged for the end-state walk
    int redone;
    int flag[3];                        // relay: the neighbour's state has arrived ([0] forward, [1] backward, [2] Viterbi)
};

__device__ __forceinline__ void lp_fwd_step(double& a0, double& a1, const double2 le, const KScalars& ks, uint32_t lut)
{
    // a[i][t] = LSE_k(lt[k][i] + a[k][t-1]) + le[i][aa[t]], k ascending (:3359-3367)
    const double f0 = lse_lut2<false>(ks.lt00 + a0, ks.lt10 + a1, lut) + le.x;
    const double f1 = lse_lut2<false>(ks.lt01 + a0, ks.lt11 + a1, lut) + le.y;
    a0 = f0;
    a1 = f1;
}
__device__ __forceinline__ void lp_bwd_step(double& b0, double& b1, const double2 le_next, const KScalars& ks, uint32_t lut)
{
    // b[i][t] = LSE_k((lt[i][k] + b[k][t+1]) + le[k][aa[t+1]]), k ascending (:3384-3389)
    const double x0 = (ks.lt00 + b0) + le_next.x, x1 = (ks.lt01 + b1) + le_next.y;
    const double y0 = (ks.lt10 + b0) + le_next.x, y1 = (ks.lt11 + b1) + le_next.y;
    b0 = lse_lut2<false>(x0, x1, lut);
    b1 = lse_lut2<false>(y0, y1, lut);
}
// ulp of the binade of |x| (|x| >= 1024 wherever this is used)
__device__ __forceinline__ double lp_ulp(double x)
{
    return __hiloint2double((((__double2hiint(fabs(x)) >> 20) & 0x7ff) - 52) << 20, 0);
}
// does a value that moves between lo_v and hi_v (any order) leave its binade, margin included?
__device__ __forceinline__ bool lp_cross(double v0, double v1)
{
    const double lo = fmin(fabs(v0), fabs(v1)) - 64.0, hi = fmax(fabs(v0), fabs(v1)) + 64.0;
    return !(lo >= 1024.0) || (__double2hiint(lo) >> 20) != (__double2hiint(hi) >> 20);
}
// Explicit shared-memory accesses for the carry walkers: nvcc forms the address of the dynamic shared segment from
// SR_CgaCtaId and, under register pressure (the kernel sits at 128 registers), re-reads that special register in front of
// accesses inside the walkers' loops.  An address laundered through an asm statement stays in a register (carry phase at
// 100 k residues: 848 k -> 693 k cycles).
__device__ __forceinline__ double lp_lds(uint32_t a)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lp_lds_u8(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void lp_sts(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void lp_sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
// message passing between the walkers of neighbouring CTAs: payload, cluster-scope fence, flag
__device__ __forceinline__ void lp_signal(int* remote_flag)
{
    asm volatile("fence.acq_rel.cluster;" ::: "memory");
    *reinterpret_cast<volatile int*>(remote_flag) = 1;
}
__device__ __forceinline__ void lp_wait(int* flag)
{
    while (*reinterpret_cast<volatile int*>(flag) == 0) __nanosleep(128);
    asm volatile("fence.acq_rel.cluster;" ::: "memory");
}
#define LP_OFF(member) ((uint32_t)offsetof(LpShared, member))

// Wherever a few lanes of a CTA work while the rest waits (scans, the carry walkers), the CTA meets at its own barrier
// before it goes to the cluster barrier: threads parked at bar.sync do not issue (carry phase at 100 k residues with the
// waiting warps at the cluster barrier: 1 010 k cycles, at the CTA barrier: 848 k).
__device__ __forceinline__ void lp_cluster_sync(cg::cluster_group& cluster)
{
    __syncthreads();
    cluster.sync();
}
struct LpMP {  // 2x2 max-plus matrix
    double m00, m01, m10, m11;
};
__device__ __forceinline__ LpMP lp_mp_mul(const LpMP& a, const LpMP& b)
{
    LpMP r;  // (a (x) b)[i][e] = max_m a[i][m] + b[m][e]
    r.m00 = fmax(a.m00 + b.m00, a.m01 + b.m10);
    r.m01 = fmax(a.m00 + b.m01, a.m01 + b.m11);
    r.m10 = fmax(a.m10 + b.m00, a.m11 + b.m10);
    r.m11 = fmax(a.m10 + b.m01, a.m11 + b.m11);
    return r;
}

__global__ void __launch_bounds__(kLpThreads, 1) k_long_post(LongPostArgs g)
{
    cg::cluster_group cluster = cg::this_cluster();
    const int X = g.cluster;
    const int pslot = blockIdx.x / X;
    const int rank = (int)cluster.block_rank();
    const int32_t prot = g.list[pslot];
    const int64_t o = g.offsets[prot];
    const int n = (int)(g.offsets[prot + 1] - o);
    // size classes: the whole cluster leaves together
    if ((X > 1) != (n >= g.big_min)) return;

    extern __shared__ __align__(16) unsigned char lp_smem[];
    LpShared& sm = *reinterpret_cast<LpShared*>(lp_smem);
    const KScalars& ks = g.ks;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint8_t* __restrict__ src = g.codes + (o - g.off_base);
    const int64_t so = g.scratch_off[pslot];
    double* __restrict__ S0 = g.S0 + so;
    double* __restrict__ S1 = g.S1 + so;
    double* __restrict__ gA = g.bnd + (so >> 5);                     // gA[j]: approximate a0 at residue j*C - 1 (j = 1..K)
    double* __restrict__ gB = gA + g.bnd_plane;                      // gB[j]: approximate b0 at residue j*C     (j = 0..K-1)
    double* __restrict__ gV0 = gA + 2 * g.bnd_plane;                 // gV*[k]: approximate Viterbi scores at chunk k's last residue
    double* __restrict__ gV1 = gA + 3 * g.bnd_plane;
    unsigned char* __restrict__ gC = reinterpret_cast<unsigned char*>(gA + 4 * g.bnd_plane);  // per chunk: choice | cross << 2; [K]: vlast
    uint8_t* __restrict__ tb = g.tb + so;
    const bool vit = g.want_vit != 0;
    const bool post = g.want_post != 0;

    // geometry: C residues per chunk, K chunks over the cluster's lanes, warm-up of m whole chunks
    const int lanes = X * kLpThreads;
    const int C = max(kLpMinChunk, (n + lanes - 1) / lanes);
    const int K = (n + C - 1) / C;
    const int m = (max(1, g.warm) + C - 1) / C;
    const int R = (K + kLpThreads - 1) / kLpThreads;  // CTAs that own chunks

    {
        const DeviceTables* T = g.tabs;
        for (int i = tid; i <= PLAAC_LUT_LEN; i += kLpThreads) {
            const double l0 = i < PLAAC_LUT_LEN ? T->lut[i] : 0.0;
            const double l1 = i + 1 < PLAAC_LUT_LEN ? T->lut[i + 1] : 0.0;
            sm.lut2[i] = make_double2(l0, l1);
        }
        if (tid < 32) sm.le[tid] = make_double2(T->le0[tid], T->le1[tid]);
        if (tid == 0) sm.redone = 0, sm.flag[0] = sm.flag[1] = sm.flag[2] = 0;
    }
    __syncthreads();
    const uint32_t lut = smem_u32(&sm.lut2[0]);
    uint32_t sbase;
    asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"(smem_u32(lp_smem)));
    // invalid input (> 21) is scored as X, as everywhere else (reported by k_pack)
    auto LE = [&](int t) -> double2 {
        const uint32_t c = src[t];
        return sm.le[c > 21u ? 0u : c];
    };

    const int kg = rank * kLpThreads + tid;  // this lane's chunk
    const bool live = kg < K;
    const int cs = kg * C, ce = min(n, cs + C);
    const int m2 = min(m, (kLpWarm2 + C - 1) / C);
    // forward: state initialised AT residue fi (true init when fi == 0), first step at fi + 1; pass 2 starts AT fi2 >= fi
    const int fi = (kg - m <= 0) ? 0 : (kg - m) * C - 1;
    const int fi2 = (kg - m2 <= 0) ? 0 : (kg - m2) * C - 1;
    // backward: state initialised AT residue bi (true init when bi == n-1), first step at bi - 1; pass 2 starts AT bi2 <= bi
    const int bi = (kg + m + 1 >= K) ? n - 1 : (kg + m + 1) * C;
    const int bi2 = (kg + m2 + 1 >= K) ? n - 1 : (kg + m2 + 1) * C;

    // ================= pass 1: chunk-local frame =================
    // From a generic start d = x1 - x0 needs ~130-190 residues to coalesce (measured: 2 of 3125 chunks fail with 128,
    // none with 192).  A lane whose warm-up reaches the protein's start (end) runs the TRUE chain: its boundary states are
    // exact as they are (mode 2).  The others keep d and the local x0 at the start of pass 2's short warm-up.
    double fw_x = 0, fw_d = 0, fw_e = 0, bw_x = 0, bw_d = 0, bw_e = 0;
    if (live) {
        {
            const double2 l0 = LE(fi);
            double a0 = ks.li0 + l0.x, a1 = ks.li1 + l0.y, e0 = 0.0, e1 = 0.0;
            if (fi2 == fi) fw_x = a0, fw_d = a1 - a0;
#pragma unroll 4
            for (int t = fi + 1; t < ce; t++) {
                if (t == cs) e0 = a0, e1 = a1;
                lp_fwd_step(a0, a1, LE(t), ks, lut);
                if (t == fi2) fw_x = a0, fw_d = a1 - a0;
            }
            fw_e = e0;
            sm.inc[0][tid] = a0 - e0;  // first chunk: e0 = 0, absolute
            if (fi == 0) {
                sm.mode[0][tid] = 2;
                sm.g_ea0[0][0][tid] = e0, sm.g_den[0][0][tid] = e1;
                sm.g_ea0[0][1][tid] = a0, sm.g_den[0][1][tid] = a1;
            }
        }
        if (!post) {
            sm.inc[1][tid] = 0.0;
            sm.mode[1][tid] = 1;
        } else {
            double b0 = ks.lf0, b1 = ks.lf1, e0 = 0.0, e1 = 0.0;
            if (bi2 == bi) bw_x = b0, bw_d = b1 - b0;
#pragma unroll 4
            for (int t = bi - 1; t >= cs; t--) {
                if (t == ce - 1) e0 = b0, e1 = b1;
                lp_bwd_step(b0, b1, LE(t + 1), ks, lut);
                if (t == bi2) bw_x = b0, bw_d = b1 - b0;
            }
            bw_e = e0;
            sm.inc[1][tid] = b0 - e0;  // last chunk: e0 = 0, absolute
            if (bi == n - 1) {
                sm.mode[1][tid] = 2;
                sm.g_ea0[1][0][tid] = e0, sm.g_den[1][0][tid] = e1;
                sm.g_ea0[1][1][tid] = b0, sm.g_den[1][1][tid] = b1;
            }
        }
        if (vit) {
            // Viterbi: the chunk's max-plus transfer matrix from both unit start vectors (first chunk: the true chain with
            // its traceback bits -- row 1 of its "matrix" is -Inf, so row 0 of every prefix product is the score vector)
            double a0 = 0.0, a1 = -INFINITY, b0 = -INFINITY, b1 = 0.0;
            int t0 = cs;
            if (kg == 0) {
                const double2 l0 = LE(0);
                a0 = ks.li0 + l0.x, a1 = ks.li1 + l0.y, b1 = -INFINITY;
                tb[0] = 0;
                t0 = 1;
            }
#pragma unroll 4
            for (int t = t0; t < ce; t++) {
                const double2 le = LE(t);
                const double vA00 = ks.lt00 + a0, vA10 = ks.lt10 + a1, vA01 = ks.lt01 + a0, vA11 = ks.lt11 + a1;
                const double vB00 = ks.lt00 + b0, vB10 = ks.lt10 + b1, vB01 = ks.lt01 + b0, vB11 = ks.lt11 + b1;
                const bool pA0 = vA10 > vA00, pA1 = vA11 > vA01;
                a0 = (pA0 ? vA10 : vA00) + le.x;
                a1 = (pA1 ? vA11 : vA01) + le.y;
                b0 = fmax(vB00, vB10) + le.x;
                b1 = fmax(vB01, vB11) + le.y;
                if (kg == 0) tb[t] = (uint8_t)((int)pA0 | ((int)pA1 << 1));
            }
            sm.vMi[tid][0] = a0, sm.vMi[tid][1] = a1, sm.vMi[tid][2] = b0, sm.vMi[tid][3] = b1;
            if (kg == 0) sm.vE0 = a0, sm.vE1 = a1;
        }
    } else {
        sm.inc[0][tid] = 0.0;
        sm.inc[1][tid] = 0.0;
        sm.vMi[tid][0] = 0.0, sm.vMi[tid][1] = -INFINITY, sm.vMi[tid][2] = -INFINITY, sm.vMi[tid][3] = 0.0;  // identity
    }
    __syncthreads();
    if (vit && wid == 2) {
        // inclusive prefix products of the chunk matrices (Kogge-Stone over warp shuffles, carry across the rounds)
        LpMP c = {0.0, -INFINITY, -INFINITY, 0.0};
        for (int r = 0; r < kLpThreads / 32; r++) {
            const int idx = r * 32 + lane;
            LpMP p = {sm.vMi[idx][0], sm.vMi[idx][1], sm.vMi[idx][2], sm.vMi[idx][3]};
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                LpMP q;
                q.m00 = __shfl_up_sync(0xffffffffu, p.m00, d), q.m01 = __shfl_up_sync(0xffffffffu, p.m01, d);
                q.m10 = __shfl_up_sync(0xffffffffu, p.m10, d), q.m11 = __shfl_up_sync(0xffffffffu, p.m11, d);
                if (lane >= d) p = lp_mp_mul(q, p);
            }
            p = lp_mp_mul(c, p);
            sm.vMi[idx][0] = p.m00, sm.vMi[idx][1] = p.m01, sm.vMi[idx][2] = p.m10, sm.vMi[idx][3] = p.m11;
            c.m00 = __shfl_sync(0xffffffffu, p.m00, 31), c.m01 = __shfl_sync(0xffffffffu, p.m01, 31);
            c.m10 = __shfl_sync(0xffffffffu, p.m10, 31), c.m11 = __shfl_sync(0xffffffffu, p.m11, 31);
        }
        if (lane == 0) sm.vtot[0] = c.m00, sm.vtot[1] = c.m01, sm.vtot[2] = c.m10, sm.vtot[3] = c.m11;
    }
    // local scans: warp 0 inclusive prefix of the forward increments, warp 1 inclusive suffix of the backward ones
    if (wid < 2) {
        double carry = 0.0;
        for (int r = 0; r < kLpThreads / 32; r++) {
            const int idx = wid == 0 ? r * 32 + lane : kLpThreads - 1 - (r * 32 + lane);
            double v = sm.inc[wid][idx];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double u = __shfl_up_sync(0xffffffffu, v, d);
                if (lane >= d) v += u;
            }
            v += carry;
            sm.inc[wid][idx] = v;
            carry = __shfl_sync(0xffffffffu, v, 31);
        }
        if (lane == 0) sm.tot[wid] = carry;
    }
    lp_cluster_sync(cluster);
    {
        // cross-CTA carry of the approximate sums through distributed shared memory
        double offF = 0.0, offB = 0.0;
        for (int r = 0; r < X; r++) {
            const double* t = cluster.map_shared_rank(&sm.tot[0], r);
            if (r < rank) offF += t[0];
            if (r > rank) offB += t[1];
        }
        if (live) {
            gA[kg + 1] = offF + sm.inc[0][tid];
            gB[kg] = offB + sm.inc[1][tid];
        }
        if (vit) {
            LpMP cin = {0.0, -INFINITY, -INFINITY, 0.0};
            for (int r = 0; r < rank; r++) {
                const double* t = cluster.map_shared_rank(&sm.vtot[0], r);
                const LpMP m = {t[0], t[1], t[2], t[3]};
                cin = lp_mp_mul(cin, m);
            }
            if (live) {
                gV0[kg] = fmax(cin.m00 + sm.vMi[tid][0], cin.m01 + sm.vMi[tid][2]);
                gV1[kg] = fmax(cin.m00 + sm.vMi[tid][1], cin.m01 + sm.vMi[tid][3]);
            }
        }
    }
    lp_cluster_sync(cluster);

    // ================= pass 2: the jar's own binade, two frames one ulp apart =================
    if (live) {
        // ---- forward (frames start AT fi2 with pass 1's d and the approximate absolute x0 there)
        if (fi != 0) {
            if (lp_cross(gA[kg], gA[kg + 1])) {
                sm.mode[0][tid] = 1;
            } else {
                const double u = lp_ulp(gA[kg]);
                double a0 = gA[kg] - (fw_e - fw_x), a1 = a0 + fw_d, c0 = a0 + u, c1 = c0 + fw_d;
                double ea = 0, ed = 0, ec = 0, ee = 0;
#pragma unroll 2
                for (int t = fi2 + 1; t < ce; t++) {
                    if (t == cs) {
                        ea = a0, ed = a1 - a0;
                        ec = c0, ee = c1 - c0;
                    }
                    const double2 le = LE(t);
                    lp_fwd_step(a0, a1, le, ks, lut);
                    lp_fwd_step(c0, c1, le, ks, lut);
                }
                sm.mode[0][tid] = 0;
                sm.g_inc[0][0][tid] = a0 - ea, sm.g_ea0[0][0][tid] = ea, sm.g_den[0][0][tid] = ed, sm.g_dex[0][0][tid] = a1 - a0;
                sm.g_inc[0][1][tid] = c0 - ec, sm.g_ea0[0][1][tid] = ec, sm.g_den[0][1][tid] = ee, sm.g_dex[0][1][tid] = c1 - c0;
            }
        }
        // ---- backward
        if (post && bi != n - 1) {
            if (lp_cross(gB[kg + 1], gB[kg])) {
                sm.mode[1][tid] = 1;
            } else {
                const double u = lp_ulp(gB[kg + 1]);
                double a0 = gB[kg + 1] - (bw_e - bw_x), a1 = a0 + bw_d, c0 = a0 + u, c1 = c0 + bw_d;
                double ea = 0, ed = 0, ec = 0, ee = 0;
#pragma unroll 2
                for (int t = bi2 - 1; t >= cs; t--) {
                    if (t == ce - 1) {
                        ea = a0, ed = a1 - a0;
                        ec = c0, ee = c1 - c0;
                    }
                    const double2 le = LE(t + 1);
                    lp_bwd_step(a0, a1, le, ks, lut);
                    lp_bwd_step(c0, c1, le, ks, lut);
                }
                sm.mode[1][tid] = 0;
                sm.g_inc[1][0][tid] = a0 - ea, sm.g_ea0[1][0][tid] = ea, sm.g_den[1][0][tid] = ed, sm.g_dex[1][0][tid] = a1 - a0;
                sm.g_inc[1][1][tid] = c0 - ec, sm.g_ea0[1][1][tid] = ec, sm.g_den[1][1][tid] = ee, sm.g_dex[1][1][tid] = c1 - c0;
            }
        }
        // both frames tell the same story?  (entries an odd number of ulps apart: one of them has the right parity)
#pragma unroll
        for (int dir = 0; dir < 2; dir++) {
            bool ty = false;
            if (sm.mode[dir][tid] == 0) {
                const double u = lp_ulp(sm.g_ea0[dir][0][tid]);
                const double q = (sm.g_ea0[dir][1][tid] - sm.g_ea0[dir][0][tid]) / u;
                ty = __double_as_longlong(sm.g_den[dir][0][tid]) == __double_as_longlong(sm.g_den[dir][1][tid]) &&
                     __double_as_longlong(sm.g_dex[dir][0][tid]) == __double_as_longlong(sm.g_dex[dir][1][tid]) &&
                     sm.g_inc[dir][0][tid] == sm.g_inc[dir][1][tid] && fabs(q) < 1e6 && q == rint(q) && q != 2.0 * rint(0.5 * q);
            }
            sm.typ[dir][tid] = ty ? 1 : 0;
        }
        if (vit && kg >= 1) {
            // Viterbi in the jar's binade: entered with score R in state 0 (frame A) or in state 1 (frame B); the exact
            // entry scores differ from R by exact shifts, which commute with every rounding of the chunk
            const double p0 = gV0[kg - 1], p1 = gV1[kg - 1];
            const double lo = fmin(fabs(p0), fabs(p1)) - 64.0, hi = fmax(fabs(gV0[kg]), fabs(gV1[kg])) + 64.0;
            const bool cross = !(lo >= 1024.0) || (__double2hiint(lo) >> 20) != (__double2hiint(hi) >> 20) ||
                               ((g.vit_tie_mask >> (((__double2hiint(lo) >> 20) & 0x7ff) - 1023)) & 1ull);
            sm.vcross[tid] = cross ? 1 : 0;
            if (!cross) {
                const double R = p0;
                double a0 = R, a1 = -INFINITY, b0 = -INFINITY, b1 = R;
#pragma unroll 4
                for (int t = cs; t < ce; t++) {
                    const double2 le = LE(t);
                    const double vA00 = ks.lt00 + a0, vA10 = ks.lt10 + a1, vA01 = ks.lt01 + a0, vA11 = ks.lt11 + a1;
                    const double vB00 = ks.lt00 + b0, vB10 = ks.lt10 + b1, vB01 = ks.lt01 + b0, vB11 = ks.lt11 + b1;
                    const bool pA0 = vA10 > vA00, pA1 = vA11 > vA01, pB0 = vB10 > vB00, pB1 = vB11 > vB01;
                    a0 = (pA0 ? vA10 : vA00) + le.x;
                    a1 = (pA1 ? vA11 : vA01) + le.y;
                    b0 = (pB0 ? vB10 : vB00) + le.x;
                    b1 = (pB1 ? vB11 : vB01) + le.y;
                    tb[t] = (uint8_t)((int)pA0 | ((int)pA1 << 1) | ((int)pB0 << 2) | ((int)pB1 << 3));
                }
                // relative to the entry score: exact differences (one binade), so the walker's S + (M - R) is its (S - R) + M
                sm.vMi[tid][0] = a0 - R, sm.vMi[tid][1] = a1 - R, sm.vMi[tid][2] = b0 - R, sm.vMi[tid][3] = b1 - R;
            }
        } else if (vit) {
            sm.vcross[tid] = 0;  // first chunk: the true chain of pass 1 (vE0, vE1)
        }
    } else {
        sm.typ[0][tid] = sm.typ[1][tid] = 0;
        sm.mode[0][tid] = sm.mode[1][tid] = 1;
    }
    lp_cluster_sync(cluster);
    // link to the chunk before this one in walking order (the neighbour lane, or the neighbour CTA's edge lane over DSMEM)
    {
#pragma unroll
        for (int dir = 0; dir < 2; dir++) {
            bool lk = false;
            const int kp = dir == 0 ? kg - 1 : kg + 1;
            if (live && sm.typ[dir][tid] && kp >= 0 && kp < K) {
                const int rp = kp / kLpThreads, lp = kp % kLpThreads;
                const LpShared* o = rp == rank ? &sm : cluster.map_shared_rank(&sm, rp);
                lk = o->typ[dir][lp] && __double_as_longlong(o->g_dex[dir][0][lp]) == __double_as_longlong(sm.g_den[dir][0][tid]);
            }
            sm.link[dir][tid] = lk ? 1 : 0;
        }
    }
    lp_cluster_sync(cluster);

    // ================= carry: exact state at every chunk boundary, in chunk order, relayed over the cluster =================
    // One lane per chain (forward, backward, Viterbi) on three different warps.  The values of the next chunk are loaded
    // while the current one is added: the dependent chain of the common case is one fp64 addition per chunk.
    {
        if (vit && tid == 64 && rank < R) {
            if (rank > 0) lp_wait(&sm.flag[2]);
            // exact Viterbi scores in chunk order (first strict maximum as in :3090-3099), choice bits per chunk
            const int k_lo = rank * kLpThreads, k_hi = min(K, k_lo + kLpThreads);
            double Sx0 = *reinterpret_cast<volatile double*>(&sm.vcarry[0]), Sx1 = *reinterpret_cast<volatile double*>(&sm.vcarry[1]);
            const uint32_t aM = sbase + LP_OFF(vMi), aX = sbase + LP_OFF(vcross), aCh = sbase + LP_OFF(vchoice);
            int k = k_lo;
            if (k == 0) {  // the first chunk is the true chain of pass 1
                Sx0 = sm.vE0, Sx1 = sm.vE1;
                lp_sts_u8(aCh, 0u);
                k = 1;
            }
            double2 nA = make_double2(0.0, 0.0), nB = nA;
            uint32_t ncr = 0;
            if (k < k_hi) {
                nA = lds_v2f64(aM + (uint32_t)(k - k_lo) * 32u), nB = lds_v2f64(aM + (uint32_t)(k - k_lo) * 32u + 16u);
                ncr = lp_lds_u8(aX + (uint32_t)(k - k_lo));
            }
            for (; k < k_hi; k++) {
                const int l = k - k_lo;
                const double M0 = nA.x, M1 = nA.y, M2 = nB.x, M3 = nB.y;
                const uint32_t cr = ncr;
                if (k + 1 < k_hi) {
                    const uint32_t o32 = (uint32_t)(l + 1) * 32u;
                    nA = lds_v2f64(aM + o32), nB = lds_v2f64(aM + o32 + 16u);
                    ncr = lp_lds_u8(aX + (uint32_t)(l + 1));
                }
                if (cr) {
                    const int s = k * C, e = min(n, s + C);
                    int f0 = 0, f1 = 1;  // state at the last residue of the previous chunk if the state at t is 0 / 1
#pragma unroll 4
                    for (int t = s; t < e; t++) {
                        const double2 le = LE(t);
                        const double v00 = ks.lt00 + Sx0, v10 = ks.lt10 + Sx1, v01 = ks.lt01 + Sx0, v11 = ks.lt11 + Sx1;
                        const bool p0 = v10 > v00, p1 = v11 > v01;
                        Sx0 = (p0 ? v10 : v00) + le.x;
                        Sx1 = (p1 ? v11 : v01) + le.y;
                        tb[t] = (uint8_t)((int)p0 | ((int)p1 << 1));
                        const int m0 = p0 ? f1 : f0, m1 = p1 ? f1 : f0;
                        f0 = m0, f1 = m1;
                    }
                    lp_sts_u8(aCh + (uint32_t)l, (uint32_t)(f0 | (f1 << 1)));
                } else {
                    const double x00 = Sx0 + M0, x10 = Sx1 + M2;  // exact: M holds the chunk's transfer entries relative to R
                    const double x01 = Sx0 + M1, x11 = Sx1 + M3;
                    const int ch0 = x10 > x00 ? 1 : 0, ch1 = x11 > x01 ? 1 : 0;
                    Sx0 = ch0 ? x10 : x00;
                    Sx1 = ch1 ? x11 : x01;
                    lp_sts_u8(aCh + (uint32_t)l, (uint32_t)(ch0 | (ch1 << 1)));
                }
            }
            if (rank + 1 < R) {
                LpShared* o = cluster.map_shared_rank(&sm, rank + 1);
                *reinterpret_cast<volatile double*>(&o->vcarry[0]) = Sx0;
                *reinterpret_cast<volatile double*>(&o->vcarry[1]) = Sx1;
                lp_signal(&o->flag[2]);
            } else {
                const double e0v = Sx0 + ks.lf0, e1v = Sx1 + ks.lf1;  // :3102-3108
                gC[K] = (unsigned char)(e1v > e0v ? 1 : 0);
                if (g.hmm_out) g.hmm_out[2 * pslot + 1] = e1v > e0v ? e1v : e0v;
            }
        }
        const int dir = (tid == 0) ? 0 : ((tid == 32 && post) ? 1 : -1);
        if (dir >= 0 && rank < R) {
            const bool first = dir == 0 ? rank == 0 : rank == R - 1;
            if (!first) lp_wait(&sm.flag[dir]);
            const int k_lo = rank * kLpThreads, k_hi = min(K, k_lo + kLpThreads);  // this CTA's chunks
            const int cnt = k_hi - k_lo, l_first = dir == 0 ? 0 : cnt - 1, l_step = dir == 0 ? 1 : -1;
            double x0 = *reinterpret_cast<volatile double*>(&sm.carry[dir][0]);   // (unused by the first walker)
            double x1 = *reinterpret_cast<volatile double*>(&sm.carry[dir][1]);
            bool acc = !first && *reinterpret_cast<volatile int*>(&sm.carry_acc[dir]) != 0;  // the chunk before was accepted with its frames
            int nredo = 0;
            const uint32_t aL = sbase + LP_OFF(link) + (uint32_t)dir * kLpThreads;
            const uint32_t aI = sbase + LP_OFF(g_inc) + (uint32_t)dir * 2u * kLpThreads * 8u;  // [dir][0][.]
            const uint32_t aD = sbase + LP_OFF(g_dex) + (uint32_t)dir * 2u * kLpThreads * 8u;
            const uint32_t aE0 = sbase + LP_OFF(ent0) + (uint32_t)dir * kLpThreads * 8u, aE1 = sbase + LP_OFF(ent1) + (uint32_t)dir * kLpThreads * 8u;
            uint32_t nlk = lp_lds_u8(aL + (uint32_t)l_first);
            double ninc = lp_lds(aI + (uint32_t)l_first * 8u), ndex = lp_lds(aD + (uint32_t)l_first * 8u);
            for (int q = 0; q < cnt; q++) {
                const int l = l_first + q * l_step, k = k_lo + l;
                const uint32_t lk = nlk;
                const double inc = ninc, dexo = ndex;
                if (q + 1 < cnt) {
                    const uint32_t ln = (uint32_t)(l + l_step);
                    nlk = lp_lds_u8(aL + ln);
                    ninc = lp_lds(aI + ln * 8u);
                    ndex = lp_lds(aD + ln * 8u);
                }
                lp_sts(aE0 + (uint32_t)l * 8u, x0);
                lp_sts(aE1 + (uint32_t)l * 8u, x1);
                if (lk && acc) {
                    x0 = x0 + inc;
                    x1 = x0 + dexo;
                    continue;
                }
                const int md = sm.mode[dir][l];
                if (md == 2) {
                    x0 = sm.g_ea0[dir][1][l];
                    x1 = sm.g_den[dir][1][l];
                    acc = false;
                    continue;
                }
                int fr = -1;
                if (md == 0) {
                    const double u = lp_ulp(x0);
                    const double dex = x1 - x0;
#pragma unroll
                    for (int f = 0; f < 2; f++) {
                        const double qd = (sm.g_ea0[dir][f][l] - x0) / u;  // exact: a small integer
                        if (fr < 0 && qd == 2.0 * rint(0.5 * qd) &&
                            __double_as_longlong(sm.g_den[dir][f][l]) == __double_as_longlong(dex))
                            fr = f;
                    }
                }
                if (fr >= 0) {
                    x0 = x0 + sm.g_inc[dir][fr][l];
                    x1 = x0 + sm.g_dex[dir][fr][l];
                    acc = true;  // (links are only set behind typ chunks: either frame's exit d is the chunk's)
                } else {
                    const int s = k * C, e = min(n, s + C);
                    if (dir == 0) {
#pragma unroll 4
                        for (int t = s; t < e; t++) lp_fwd_step(x0, x1, LE(t), ks, lut);
                    } else {
#pragma unroll 4
                        for (int t = e - 1; t >= s; t--) lp_bwd_step(x0, x1, LE(t + 1), ks, lut);
                    }
                    nredo += md == 0 ? 1 : 0;
                    acc = false;
                }
            }
            if (nredo) atomicAdd(&sm.redone, nredo);
            // hand the exact state to the neighbour
            const int next = dir == 0 ? rank + 1 : rank - 1;
            if (next >= 0 && next < R) {
                LpShared* o = cluster.map_shared_rank(&sm, next);
                *reinterpret_cast<volatile double*>(&o->carry[dir][0]) = x0;
                *reinterpret_cast<volatile double*>(&o->carry[dir][1]) = x1;
                *reinterpret_cast<volatile int*>(&o->carry_acc[dir]) = acc ? 1 : 0;
                lp_signal(&o->flag[dir]);
            } else if (dir == 0 && g.hmm_out) {
                g.hmm_out[2 * pslot] = lse_lut2<false>(x0 + ks.lf0, x1 + ks.lf1, lut);  // lmarginalprob :3369-3375
            }
        }
        __syncthreads();  // (the other lanes sleep here; the waiting walkers of other CTAs poll their flags with back-off)
    }
    if (vit) {
        // every CTA publishes its chunks' choice bytes (choice | cross << 2)
        if (live) gC[kg] = (unsigned char)(sm.vchoice[tid] | (sm.vcross[tid] << 2));
        __threadfence();
        lp_cluster_sync(cluster);
    }

    // ================= pass 3: every chunk from its exact boundary state =================
    if (live && post) {
        {
            double b0, b1;
            int t = ce - 1;
            if (kg == K - 1) {
                b0 = ks.lf0, b1 = ks.lf1;  // :3379-3381
                S0[n - 1] = b0;
                S1[n - 1] = b1;
                t = n - 2;
            } else {
                b0 = sm.ent0[1][tid], b1 = sm.ent1[1][tid];
            }
#pragma unroll 4
            for (; t >= cs; t--) {
                lp_bwd_step(b0, b1, LE(t + 1), ks, lut);
                S0[t] = b0;
                S1[t] = b1;
            }
        }
        {
            double a0, a1;
            int t = cs;
            if (kg == 0) {
                const double2 l0 = LE(0);
                a0 = ks.li0 + l0.x, a1 = ks.li1 + l0.y;  // :3356-3358
                const double s0 = a0 + S0[0], s1 = a1 + S1[0];
                g.lpseq[pslot] = lse_lut2<false>(s0, s1, lut);  // :3393-3396
                S0[0] = s0;
                S1[0] = s1;
                t = 1;
            }  else {
                a0 = sm.ent0[0][tid], a1 = sm.ent1[0][tid];
            }
            // b of four residues is fetched (L2) before the four steps that use it
            for (; t < ce; t += 4) {
                double s0v[4], s1v[4];
                double2 lev[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int tt = min(t + u, ce - 1);
                    s0v[u] = S0[tt];
                    s1v[u] = S1[tt];
                    lev[u] = LE(tt);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (t + u < ce) {
                        lp_fwd_step(a0, a1, lev[u], ks, lut);
                        S0[t + u] = a0 + s0v[u];
                        S1[t + u] = a1 + s1v[u];
                    }
                }
            }
        }
    }
    if (vit) {
        // State at the last residue of every chunk: endstate[k-1] = choice[k](endstate[k]), a suffix composition of 2 -> 2
        // maps.  One warp: lane j composes the maps of its block of chunks, the lanes are chained, the block is walked again.
        for (int k = tid; k <= K; k += kLpThreads) sm.vall[k] = gC[k];
        __syncthreads();
        if (wid == 3 && rank < R) {
            const int B = (K + 31) / 32;
            const int hi = min(K, (lane + 1) * B) - 1, lo = lane * B;   // this lane's chunks, walked from hi down to lo
            // composite map of the block: state above the block (at chunk hi) -> state at chunk lo - 1
            int f0 = 0, f1 = 1;
            for (int k = hi; k >= lo; k--) {
                const int c = sm.vall[k];
                f0 = (c >> f0) & 1;
                f1 = (c >> f1) & 1;
            }
            // state at this lane's top chunk: vlast pushed through the blocks above
            int e = sm.vall[K];
            for (int j = 31; j >= 1; j--) {  // (uniform trip count: every lane takes part in every shuffle)
                const int g0 = __shfl_sync(0xffffffffu, f0, j), g1 = __shfl_sync(0xffffffffu, f1, j);
                if (j > lane && j * B < K) e = e ? g1 : g0;
            }
            const int k_lo = rank * kLpThreads;
            for (int k = hi; k >= lo; k--) {
                if (k >= k_lo && k < k_lo + kLpThreads) sm.vend[k - k_lo] = (unsigned char)e;
                e = (sm.vall[k] >> e) & 1;
            }
        }
        __syncthreads();
        if (live && (g.out.vit || g.vbytes)) {
            // :3110-3113 for every chunk in parallel; frame A if the chunk is entered in state 0, B if in state 1 (redone
            // chunks and the first one hold the exact bits as frame A)
            uint8_t* dst = g.out.vit ? g.out.vit + (o - g.res_base) : g.vbytes + so;
            int v = sm.vend[tid];
            const unsigned cb = sm.vall[kg];
            const int sh = (cb & 4u) || kg == 0 ? 0 : 2 * (int)((cb >> v) & 1u);
            for (int t = ce - 1; t >= cs; t -= 8) {
                uint32_t tv[8];
#pragma unroll
                for (int u = 0; u < 8; u++) tv[u] = tb[max(t - u, cs)];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    if (t - u >= cs) {
                        dst[t - u] = (uint8_t)v;
                        v = (tv[u] >> (sh + v)) & 1;
                    }
                }
            }
        }
    }
    if (tid == 0 && sm.redone && g.redone) atomicAdd(g.redone, (unsigned long long)sm.redone);
    __threadfence();
    lp_cluster_sync(cluster);

    // ================= pass 4: posteriors and MAP bytes, coalesced =================
    if (post) {
        const double lpseq = g.lpseq[pslot];
        const int64_t ob = o - g.res_base;
        const int per = (n + X - 1) / X;
        const int t_lo = rank * per, t_hi = min(n, t_lo + per);
        bool bad = false;
        for (int t = t_lo + tid; t < t_hi; t += kLpThreads) {
            bad |= src[t] > 21;
            const double p0 = exp(S0[t] - lpseq), p1 = exp(S1[t] - lpseq);
            g.out.post_bg[ob + t] = p0;
            g.out.post_prd[ob + t] = p1;
            if (g.out.map) g.out.map[ob + t] = p1 > p0 ? 1 : 0;
        }
        if (bad && g.errflag) atomicOr(g.errflag, 1);
    }
}

}  // namespace plaac
