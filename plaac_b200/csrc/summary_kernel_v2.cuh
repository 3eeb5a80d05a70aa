// Summary-mode scoring, throughput version ("v2").
//
// One CTA = 2*NWR warps.  Warps 0..NWR-1 run role A, warps NWR..2*NWR-1 run role B, each on one length
// bucket of 32 proteins (lane = protein), all lanes advancing the residue index t in lock step:
//
//   role A (the serial recurrences, REFERENCE OPERATION ORDER, bit-faithful to plaac.java):
//     Viterbi max-plus recurrence + traceback bits   viterbidecodel :3077-3121
//     LUT forward recurrence                          posteriorl :3349-3375, logeapeb :1024-1047
//     hmm0's sequential log-emission sum              (= its Viterbi and marginal log-prob, SURVEY 8 a5)
//     sequential psum[] LLR window search             hss2 :1206-1257, call site :782-783
//     MW Q/N window (exact integers)                  :764-771
//     traceback -> Viterbi bits, longestrun           :3110-3113, :1787-1804
//     proteins whose longest PrD run reaches the core length are appended to a list for k_core_search
//   role B (sliding windows as running sums; |delta| ~1e-13, DESIGN.md "tolerances"):
//     FoldIndex runs, means                           disorderreport :4866-5068
//     PAPA centre search on the twice-smoothed tracks slidingaverage :2585-2662, :4941-4948
//     the values reported at the PAPA centre (PAPAllr, PAPAllr2) are evaluated once per protein
//
// Shared-memory traffic is the scarce resource (one 128-byte wavefront per cycle per SM), so every
// per-code table is replicated per bank group (conflict-free for any code pattern) and the 4001-entry
// log-sum-exp LUT is stored as {lut[d], lut[d+1]} pairs (one 16-byte load per lookup).  Table bases are
// aligned so that "base | code bits" forms the address in one LOP3.  Integer -> double conversions use the
// 2^52 bit trick on the FP64 pipe instead of the slow XU conversion unit.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace plaac {

constexpr int kV2MaxThreads = 768;

// Byte offsets from an 8 KB-aligned shared-memory base.
constexpr uint32_t kOffHydB = 0;         // double [64 ext codes][16 lane copies]: hydropathy on the exact-sum grid (windows)
constexpr uint32_t kOffPapB = 8192;      // double [64][16]
constexpr uint32_t kOffLlrB = 16384;     // double [64][16]   (tail loops only)
constexpr uint32_t kOffLeA = 24576;      // double2 [32 codes][8 lane copies]  {le0, le1}
constexpr uint32_t kOffLlrA = 28672;     // double [32][16]
constexpr uint32_t kOffLut2 = 32768;     // double2 [4002]  {lut[d], lut[d+1]}
constexpr uint32_t kOffHydX = kOffLut2 + (PLAAC_LUT_LEN + 1) * 16;  // double [64][16]: exact hydropathy (sequential mean)
constexpr uint32_t kV2FixedBytes = kOffHydX + 8192;
constexpr uint32_t kV2AlignSlack = 8192;

__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ double lds_f64(uint32_t addr)
{
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
template <int OFF>
__device__ __forceinline__ double lds_f64_off(uint32_t addr)
{
    double v;
    asm("ld.shared.f64 %0, [%1+%2];" : "=d"(v) : "r"(addr), "n"(OFF));
    return v;
}
__device__ __forceinline__ double2 lds_v2f64(uint32_t addr)
{
    double2 v;
    asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}

__device__ __forceinline__ double u2d(uint32_t v)
{
    // exact uint32 -> double on the FP64 pipe: 2^52 + v, minus 2^52
    return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0;
}

// logeapeb :1024-1047 for finite-or-(-Inf) arguments, given loglut[0] == ln 2 bit for bit (checked at
// plaac_create): the a == b branch (a + ln2) then equals the interpolation at c = 0.  c = |a - b| is the
// reference's (a - b) or (b - a) bit for bit; the larger argument is picked from the sign of a - b.
template <bool ALWAYS_IN>
__device__ __forceinline__ double lse_lut2(double a, double b, uint32_t lut_addr)
{
    const double d = a - b;
    const double hi = (__double2hiint(d) < 0) ? b : a;  // a == b gives +0: hi = a
    const double c = fabs(d);
    const double x = 100.0 * c;
    if (ALWAYS_IN) {
        // plaac_create proved |a - b| < 40 for every reachable argument pair of the recurrence
        // floor on the FP64 pipe: x + 2^52 rounded DOWN is 2^52 + floor(x) exactly (0 <= x < 2^51), its low word is
        // the table index and subtracting 2^52 again gives floor(x) as a double -- no F2I, no separate int -> double
        const double y = __dadd_rd(x, 4503599627370496.0);
        const double2 l = lds_v2f64(lut_addr + (uint32_t)__double2loint(y) * 16u);
        const double f1 = x - (y - 4503599627370496.0);
        const double f0 = 1.0 - f1;
        return hi + (f1 * l.y + f0 * l.x);
    }
    const bool in = c < 40.0;
    const int dex = min(__double2int_rd(x), PLAAC_LUT_LEN - 1);  // x >= 0, NaN -> 0
    const double2 l = lds_v2f64(lut_addr + (uint32_t)dex * 16u);
    const double f1 = x - u2d((uint32_t)dex);  // 100*c - dex
    const double f0 = 1.0 - f1;                // == (dex + 1) - 100*c exactly (both are exact differences)
    const double r = hi + (f1 * l.y + f0 * l.x);
    return in ? r : hi;
}

struct V2Args {
    BatchView bv;
    KScalars ks;
    const DeviceTables* tabs;
    plaac_summary* out;
    int ring_words;       // per lane, power of two
    int nwr;              // warps per role
    int32_t* core_list;   // ranks needing the CORE search
    int32_t* core_count;
    int always_in;        // 1: |a-b| < 40 is guaranteed inside the forward recurrence (bound checked on the host)
    unsigned long long* work_counter;  // zeroed before the launch
    // v3 only: host-computed (double)(2w+1)^2, cc2 * that, cc2 * (2w+1)
    double ks_wfull, ks_cc2w, ks_cc2full;
    // v3 with kV3IntFold: the FoldIndex / PAPA tests as fi_a * (sum of hydi) + fi_b * |charge| + fi_c * taps, and fi_c
    // times the unclipped tap counts 2w+1 and (2w+1)^2
    int fi_a, fi_b, fi_c, fi_cfull, fi_cw;
};

// ------------------------------------------------------------------------------------------------ role A
__device__ __forceinline__ void role_a(const V2Args& g, uint32_t sbase, uint32_t* ring, int lane, int64_t b)
{
    const KScalars& ks = g.ks;
    const BatchView& bv = g.bv;
    const int rmask = g.ring_words - 1;
    constexpr uint32_t kPadW = 0x01010101u * kPad;
    const int64_t rank = b * 32 + lane;
    int n = 0;
    int32_t prot = -1;
    if (rank < bv.nprot) {
        prot = bv.order[rank];
        n = (int)eff_len(bv.offsets[prot + 1] - bv.offsets[prot], bv.long_min);
        if (n == 0 && bv.offsets[prot + 1] != bv.offsets[prot]) prot = -1;  // scored by the long-sequence path
    }
    const int64_t cb = bv.chunk_base[b];
    const int nch = (int)(bv.chunk_base[b + 1] - cb);
    const uint4* sp = bv.stream + cb * 32 + lane;
    uint32_t* tbp = bv.tbw + cb * 32 + lane;
    const int c = ks.core_len, mw = ks.mw_window;

    const uint32_t le_base = sbase + kOffLeA + (uint32_t)(lane & 7) * 16u;
    const uint32_t ll_base = sbase + kOffLlrA + (uint32_t)(lane & 15) * 8u;
    const uint32_t lut_addr = sbase + kOffLut2;

    double s0 = 0, s1 = 0, a0 = 0, a1 = 0, sum0 = 0;
    // Sentinels: until the first complete window (t = c-1 resp. mw-1, always taken in the generic path, which
    // assigns unconditionally) no candidate can beat +Inf / INT_MAX, so the fast path needs no range test.
    double ps = 0, psl = 0, llr_best = INFINITY;
    int llr_stop = -2;
    int qn = 0, mw_best = 0x7fffffff, mw_stop = -1;
    uint32_t acc0 = 0, acc1 = 0;  // traceback bit planes, newest residue at bit 31

    // lagged byte streams: position t - off, off = 4*a + b
    const int ac = c >> 2, sc_ = 8 * (4 - (c & 3));
    const int am = mw >> 2, sm_ = 8 * (4 - (mw & 3));
    uint32_t lo_c = kPadW, lo_m = kPadW;

    uint4 nxt = make_uint4(kPadW, kPadW, kPadW, kPadW);
    if (nch > 0) nxt = sp[0];
    const int nwords = nch * 4;  // nch*16 >= nmax
    int nmin = (prot >= 0) ? n : 0x7fffffff;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) nmin = min(nmin, __shfl_xor_sync(0xffffffffu, nmin, d));
    const int wv_c1 = (c - 1) >> 2, wv_m1 = (mw - 1) >> 2;  // words holding the first complete LLR / MW window

    // one residue step; FAST: every lane has 0 < t < n-1 and t is not the first complete window of either search
    auto step = [&](auto fast_tag, auto in_tag, int t, int i, uint32_t w0, uint32_t wc, uint32_t wm) {
        constexpr bool FAST = decltype(fast_tag)::value;
        constexpr bool AIN = decltype(in_tag)::value;
        // code bits 4:0 of byte i moved to address bits 11:7
        const uint32_t k0 = (i == 0 ? (w0 << 7) : (w0 >> (8 * i - 7))) & (31u << 7);
        const uint32_t kc = (i == 0 ? (wc << 7) : (wc >> (8 * i - 7))) & (31u << 7);
        const double2 le = lds_v2f64(le_base | k0);
        const double lr0 = lds_f64(ll_base | k0);
        const double lrc = lds_f64(ll_base | kc);
        psl = psl + lrc;  // == psum[t-c+1]  (pad codes add +0.0)
        qn += (int)((ks.qn_mask >> ((w0 >> (8 * i)) & 31u)) & 1u) - (int)((ks.qn_mask >> ((wm >> (8 * i)) & 31u)) & 1u);
        uint32_t tb0u = 0, tb1u = 0;
        if (FAST || t < n) {
            if (!FAST && t == 0) {
                s0 = ks.li0 + le.x;
                s1 = ks.li1 + le.y;
                a0 = s0;
                a1 = s1;
                sum0 = le.x;
            } else {
                const double v00 = ks.lt00 + s0, v10 = ks.lt10 + s1;
                const double v01 = ks.lt01 + s0, v11 = ks.lt11 + s1;
                const bool tb0 = v10 > v00, tb1 = v11 > v01;
                s0 = (tb0 ? v10 : v00) + le.x;
                s1 = (tb1 ? v11 : v01) + le.y;
                tb0u = tb0;
                tb1u = tb1;
                const double f0 = lse_lut2<AIN>(ks.lt00 + a0, ks.lt10 + a1, lut_addr) + le.x;
                const double f1 = lse_lut2<AIN>(ks.lt01 + a0, ks.lt11 + a1, lut_addr) + le.y;
                a0 = f0;
                a1 = f1;
                sum0 = sum0 + le.x;
            }
            ps = ps + lr0;
            if (FAST || t >= c - 1) {
                const double d = ps - psl;
                if ((!FAST && t == c - 1) || d > llr_best) {
                    llr_best = d;
                    llr_stop = t;
                }
            }
            if (FAST || t >= mw - 1) {
                if ((!FAST && t == mw - 1) || qn > mw_best) {
                    mw_best = qn;
                    mw_stop = t;
                }
            } else if (t == n - 1) {
                mw_best = qn;
                mw_stop = t;
            }
        }
        acc0 = __funnelshift_r(acc0, tb0u, 1);  // after 16 steps the bit of residue 16j+i sits at 16+i
        acc1 = __funnelshift_r(acc1, tb1u, 1);
    };

#pragma unroll 1
    for (int wv = 0; wv < nwords; wv++) {
        if ((wv & 3) == 0) {
            const int j = wv >> 2;
            ring[((wv + 0) & rmask) * 32] = nxt.x;
            ring[((wv + 1) & rmask) * 32] = nxt.y;
            ring[((wv + 2) & rmask) * 32] = nxt.z;
            ring[((wv + 3) & rmask) * 32] = nxt.w;
            nxt = make_uint4(kPadW, kPadW, kPadW, kPadW);
            if (j + 1 < nch) nxt = sp[(size_t)(j + 1) * 32];
        }
        const uint32_t w0 = ring[(wv & rmask) * 32];
        const uint32_t hi_c = ring[((wv - ac) & rmask) * 32];
        const uint32_t hi_m = ring[((wv - am) & rmask) * 32];
        const uint32_t wc = __funnelshift_rc(lo_c, hi_c, sc_);
        const uint32_t wm = __funnelshift_rc(lo_m, hi_m, sm_);
        lo_c = hi_c;
        lo_m = hi_m;
        const int tbase = wv * 4;
        // warp-uniform; t = nmin-1 stays generic so the "whole protein is one MW window" case (n < mw) is seen there
        if (wv != 0 && wv != wv_c1 && wv != wv_m1 && tbase + 3 < nmin - 1) {
            if (g.always_in) {
#pragma unroll
                for (int i = 0; i < 4; i++) step(std::true_type{}, std::true_type{}, tbase + i, i, w0, wc, wm);
            } else {
#pragma unroll
                for (int i = 0; i < 4; i++) step(std::true_type{}, std::false_type{}, tbase + i, i, w0, wc, wm);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) step(std::false_type{}, std::false_type{}, tbase + i, i, w0, wc, wm);
        }
        if ((wv & 3) == 3) {
            // low half: predecessor-of-state-0 bits of the slot's 16 residues, high half: predecessor-of-state-1 bits
            tbp[(size_t)(wv >> 2) * 32] = __byte_perm(acc0, acc1, 0x7632);
        }
    }

    if (prot < 0) return;
    plaac_summary* r = g.out + prot;
    r->prot_len = n;
    if (n < 1) {
        r->mw_score = r->mw_start = r->mw_end = r->llr_start = r->llr_end = r->vit_maxrun = 0;
        r->core_start = r->core_end = r->prd_start = r->prd_end = 0;
        r->llr = r->core_score = r->prd_score = r->hmm_all = r->hmm_vit = 0;
        return;
    }
    r->mw_score = mw_best;
    r->mw_start = (n < mw) ? 0 : mw_stop - mw + 1;
    r->mw_end = mw_stop;
    if (n < c) {
        r->llr = -INFINITY;
        r->llr_start = -1;
        r->llr_end = -2;
    } else {
        r->llr = llr_best;
        r->llr_start = llr_stop - c + 1;
        r->llr_end = llr_stop;
    }
    const double e0v = s0 + ks.lf0, e1v = s1 + ks.lf1;
    const int vlast = e1v > e0v ? 1 : 0;
    const double lvit = vlast ? e1v : e0v;
    const double lmarg = lse_lut2<false>(a0 + ks.lf0, a1 + ks.lf1, lut_addr);
    r->hmm_all = lmarg - sum0;
    r->hmm_vit = lvit - sum0;

    // traceback :3110-3113 + longestrun :1787-1804, 16 residues at a time; the Viterbi bits replace the
    // traceback words.  Residue i of a slot maps the state at i to the state at i-1: f_i = (P0[i], P1[i]).
    // state_i = (f_{i+1} o ... o f_hi)(state_hi): a suffix scan of 2->2 maps (Kogge-Stone on two bit planes).
    int v = vlast, cur = 0, mx = 0;
    const int jlast = (n - 1) >> 4;
    int jhi = -1, jlo = 0;  // highest / lowest slot holding a Viterbi-1 residue
    uint32_t tw_next = tbp[(size_t)jlast * 32];
    for (int j = jlast; j >= 0; j--) {
        const uint32_t tw = tw_next;
        if (j > 0) tw_next = tbp[(size_t)(j - 1) * 32];
        const int hi = (j == jlast) ? ((n - 1) & 15) : 15;
        const uint32_t valid = (2u << hi) - 1u;  // residues 0..hi of the slot
        const uint32_t below = valid >> 1;       // residues 0..hi-1
        const uint32_t P0 = tw & 0xffffu, P1 = tw >> 16;
        uint32_t A0 = (P0 >> 1) & below;                           // S_i(0), S_i = f_{i+1} for i < hi, identity above
        uint32_t A1 = ((P1 >> 1) & below) | (0xffffu & ~below);    // S_i(1)
#pragma unroll
        for (int sft = 1; sft < 16; sft <<= 1) {
            const uint32_t B0 = A0 >> sft;                                      // S_{i+sft}, identity shifted in
            const uint32_t B1 = (A1 >> sft) | (0xffffu & ~(0xffffu >> sft));
            const uint32_t n0 = (B0 & A1) | (~B0 & A0);                         // (S_i o S_{i+sft})(0)
            const uint32_t n1 = (B1 & A1) | (~B1 & A0);
            A0 = n0;
            A1 = n1;
        }
        const uint32_t vb = (v ? A1 : A0) & valid;
        v = (int)(((vb & 1u) ? P1 : P0) & 1u);  // state of the residue before this slot
        if (vb == valid) {
            cur += hi + 1;
            mx = max(mx, cur);
        } else if (vb == 0) {
            cur = 0;
        } else {
            mx = max(mx, cur + __clz((int)~(vb << (31 - hi))));  // run entering from above continues downward
            int len = 0;
            for (uint32_t x = vb; x; x &= x >> 1) len++;
            mx = max(mx, len);
            cur = __ffs((int)~vb) - 1;  // ones at the bottom continue into the next slot
        }
        if (vb) {
            if (jhi < 0) jhi = j;
            jlo = j;
        }
        tbp[(size_t)j * 32] = vb;
    }
    r->vit_maxrun = mx;
    r->core_start = -1;
    r->core_end = -2;
    r->prd_start = -1;
    r->prd_end = -2;
    r->core_score = nan("");
    r->prd_score = 0.0;
    if (mx >= c && n >= c) {
        const int slot = atomicAdd(g.core_count, 1);
        g.core_list[2 * slot] = (int32_t)rank;
        // slots the CORE search has to visit (everything outside is masked); 16 bits each, else the whole protein
        g.core_list[2 * slot + 1] = (jhi < 65536) ? (jlo | (jhi << 16)) : (int32_t)0xffff0000;
    }
}

// ------------------------------------------------------------------------------------------------ role B
__device__ __forceinline__ void role_b(const V2Args& g, uint32_t sbase, uint32_t* ring, int lane, int64_t b)
{
    const KScalars& ks = g.ks;
    const BatchView& bv = g.bv;
    const int rmask = g.ring_words - 1;
    constexpr uint32_t kPadW = 0x01010101u * kPad;
    const int64_t rank = b * 32 + lane;
    int n = 0;
    int32_t prot = -1;
    if (rank < bv.nprot) {
        prot = bv.order[rank];
        n = (int)eff_len(bv.offsets[prot + 1] - bv.offsets[prot], bv.long_min);
        if (n == 0 && bv.offsets[prot + 1] != bv.offsets[prot]) prot = -1;  // scored by the long-sequence path
    }
    const int64_t cb = bv.chunk_base[b];
    const int nch = (int)(bv.chunk_base[b + 1] - cb);
    const uint4* sp = bv.stream + cb * 32 + lane;
    const int w = ks.w;
    const int off1 = 2 * w + 1, off2 = 4 * w + 2;
    const int a1o = off1 >> 2, s1o = 8 * (4 - (off1 & 3));
    const int a2o = off2 >> 2, s2o = 8 * (4 - (off2 & 3));
    const int full = 2 * w + 1;
    const int Wfull = full * full;
    const double cc2full = ks.cc2 * (double)full;

    const uint32_t hb = sbase + kOffHydB + (uint32_t)(lane & 15) * 8u;

    int nmax = n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, d));
    const int t_end = nmax + w;
    const int nwords = (t_end + 3) >> 2;

    double sh = 0;
    int csum = 0;
    double SLh = 0, SGh = 0, Th = 0, Dp = 0, Tp = 0;
    int SLc = 0, SGc = 0, Tac = 0;
    double Tb = 0, Wb = 1, vfib = 0;
    int pcen = -1;
    int halfw = ks.h_fi;
    if (halfw > n / 2) halfw = n / 2;
    const int fi_hi = n - halfw;     // FoldIndex scan is over p in [halfw, fi_hi)
    const int edge_hi = n - 1 - w;   // windows centred beyond this are clipped on the right
    int fi_run = 0, fi_numaa = 0, fi_maxrun = 0;  // fi_run: length of the open run of fi < 0 (snaps included)
    uint32_t lo1 = kPadW, lo2 = kPadW;
    const double WfullD = (double)Wfull;
    const double cc2W = ks.cc2 * WfullD;
    const double cc0 = ks.cc0, cc1 = ks.cc1;

    int nmin = (prot >= 0) ? n : 0x7fffffff;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) nmin = min(nmin, __shfl_xor_sync(0xffffffffu, nmin, d));
    const int fast_lo = 4 * w;  // from here on p = t-w >= 3w and k = t-2w >= 2w: no left-edge effects

    // one residue step; FAST: 4w <= t < n for every lane, so every window below is unclipped and in range
    auto step = [&](auto fast_tag, int t, int i, uint32_t w0, uint32_t w1, uint32_t w2) {
        constexpr bool FAST = decltype(fast_tag)::value;
        // ext code bits 5:0 of byte i -> address bits 12:7; charge = sign-extended bits 7:6
        const uint32_t k0 = (i == 0 ? (w0 << 7) : (w0 >> (8 * i - 7))) & (63u << 7);
        const uint32_t k1 = (i == 0 ? (w1 << 7) : (w1 >> (8 * i - 7))) & (63u << 7);
        const uint32_t k2 = (i == 0 ? (w2 << 7) : (w2 >> (8 * i - 7))) & (63u << 7);
        const int ch0 = (int)(w0 << (24 - 8 * i)) >> 30;
        const int ch1 = (int)(w1 << (24 - 8 * i)) >> 30;
        const int ch2 = (int)(w2 << (24 - 8 * i)) >> 30;
        const double hy0 = lds_f64(hb | k0), pa0 = lds_f64_off<kOffPapB>(hb | k0);
        const double hy1 = lds_f64(hb | k1), pa1 = lds_f64_off<kOffPapB>(hb | k1);
        const double hy2 = lds_f64(hb | k2), pa2 = lds_f64_off<kOffPapB>(hb | k2);
        if (FAST || t < n) {
            sh = sh + lds_f64_off<kOffHydX>(hb | k0);  // mean() :1584, sequential, exact table values
            csum += ch0;
        }
        // window sums of the zero-padded sequence: lead centre p = t-w, lag centre p-(2w+1)
        SLh = (SLh + hy0) - hy1;
        SGh = (SGh + hy1) - hy2;
        Th = (Th + SLh) - SGh;
        Dp = Dp + ((pa0 + pa2) - (pa1 + pa1));  // exact: PAPA log-odds live on a 2^-k grid
        Tp = Tp + Dp;
        SLc += ch0 - ch1;
        SGc += ch1 - ch2;
        const int aSL = abs(SLc);
        Tac += aSL - abs(SGc);
        const int p = t - w;
        // FoldIndex run scan :5010-5059 over i in [halfw, n-halfw):
        // sign of fi[p] = cc0*hydro + cc1*|charge| + cc2, scaled by the tap count (> 0)
        if (FAST) {
            const double fis = (cc0 * SLh + cc1 * u2d((uint32_t)aSL)) + cc2full;
            const bool neg = fis < 0;
            const int closed = (!neg && fi_run >= 5) ? fi_run : 0;
            fi_numaa += closed;
            fi_maxrun = max(fi_maxrun, closed);
            fi_run = neg ? fi_run + 1 : 0;
        } else if (p >= halfw && p < fi_hi) {
            double c2 = cc2full;
            if (p < w || p > edge_hi) c2 = ks.cc2 * u2d((uint32_t)(full - max(0, w - p) - max(0, p - edge_hi)));
            const double fis = (cc0 * SLh + cc1 * u2d((uint32_t)aSL)) + c2;
            const bool neg = fis < 0;
            const bool last = (p == fi_hi - 1);
            // a run that starts at the first scanned position is snapped back to residue 0,
            // one that reaches the last scanned position is snapped forward to residue n-1
            if (neg) fi_run = (fi_run == 0 && p == halfw) ? halfw + 1 : fi_run + 1;
            if (!neg || last) {
                const int len = fi_run + ((neg && last) ? (n - 1 - p) : 0);
                if (len >= 5) {
                    fi_numaa += len;
                    fi_maxrun = max(fi_maxrun, len);
                }
                fi_run = 0;
            }
        }
        // PAPA centre k = p - w: first strict maximum of Tp/W among centres with fix2 < 0 (:4941-4948)
        // Tp/Wd > Tb/Wb  <=>  Tp*Wb > Tb*Wd (both positive); products of grid units and small ints
        if (FAST) {
            const double vfi = (cc0 * Th + cc1 * u2d((uint32_t)Tac)) + cc2W;
            if ((pcen < 0 || Tp * Wb > Tb * WfullD) && vfi < 0) {
                Tb = Tp;
                Wb = WfullD;
                vfib = vfi;
                pcen = t - 2 * w;
            }
        } else {
            const int k = p - w;
            if (k >= w && k <= edge_hi) {
                double Wd = WfullD;
                if (k < 2 * w || k > edge_hi - w) {
                    const int ml = 2 * w - k, mr = k - (edge_hi - w);
                    Wd = u2d((uint32_t)(Wfull - (ml > 0 ? (ml * (ml + 1)) >> 1 : 0) - (mr > 0 ? (mr * (mr + 1)) >> 1 : 0)));
                }
                const double vfi = (cc0 * Th + cc1 * u2d((uint32_t)Tac)) + ks.cc2 * Wd;
                if ((pcen < 0 || Tp * Wb > Tb * Wd) && vfi < 0) {
                    Tb = Tp;
                    Wb = Wd;
                    vfib = vfi;
                    pcen = k;
                }
            }
        }
    };

    uint4 nxt = make_uint4(kPadW, kPadW, kPadW, kPadW);
    if (nch > 0) nxt = sp[0];
#pragma unroll 1
    for (int wv = 0; wv < nwords; wv++) {
        if ((wv & 3) == 0) {
            const int j = wv >> 2;
            ring[((wv + 0) & rmask) * 32] = nxt.x;
            ring[((wv + 1) & rmask) * 32] = nxt.y;
            ring[((wv + 2) & rmask) * 32] = nxt.z;
            ring[((wv + 3) & rmask) * 32] = nxt.w;
            nxt = make_uint4(kPadW, kPadW, kPadW, kPadW);
            if (j + 1 < nch) nxt = sp[(size_t)(j + 1) * 32];
        }
        const uint32_t w0 = ring[(wv & rmask) * 32];
        const uint32_t hi1 = ring[((wv - a1o) & rmask) * 32];
        const uint32_t hi2 = ring[((wv - a2o) & rmask) * 32];
        const uint32_t w1 = __funnelshift_rc(lo1, hi1, s1o);
        const uint32_t w2 = __funnelshift_rc(lo2, hi2, s2o);
        lo1 = hi1;
        lo2 = hi2;
        const int tbase = wv * 4;
        // warp-uniform; t <= nmin-2 keeps the last scanned FoldIndex position (p = n-1-halfw) out of the fast path
        if (tbase >= fast_lo && tbase + 3 < nmin - 1) {
#pragma unroll
            for (int i = 0; i < 4; i++) step(std::true_type{}, tbase + i, i, w0, w1, w2);
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) step(std::false_type{}, tbase + i, i, w0, w1, w2);
        }
    }

    if (prot < 0) return;
    plaac_summary* r = g.out + prot;
    if (n < 1) {
        r->fi_numaa = r->fi_maxrun = r->papa_center = 0;
        r->fi_meanhydro = r->fi_meancharge = r->fi_meancombo = 0;
        r->papa_combo = r->papa_prop = r->papa_fi = r->papa_llr = r->papa_llr2 = 0;
        return;
    }
    const double mh = (1.0 * sh) / (double)n;
    const double mc = (1.0 * (double)csum) / (double)n;
    r->fi_meanhydro = mh;
    r->fi_meancharge = mc;
    r->fi_meancombo = (ks.cc2 + ks.cc1 * fabs(mc)) + ks.cc0 * mh;
    r->fi_numaa = fi_numaa;
    r->fi_maxrun = fi_maxrun;
    r->papa_center = pcen;
    if (pcen >= 0) {
        const double prop = Tb / Wb;
        r->papa_combo = prop;
        r->papa_prop = prop;
        r->papa_fi = vfib / Wb;
        // PAPAllr = plaacllr[pcen]: 2w+1 taps in reference order (:2604-2620; pcen is interior).
        // PAPAllr2 = plaacllrx2[pcen] = sum_q (2w+1-|q-pcen|) llr[q] / W over the zero-padded sequence.
        // The 4w+1 residues around the centre are re-staged into the lane's ring column (whole 16-byte slots,
        // independent loads first), so the tap loop below reads shared memory only.
        const uint32_t lb = sbase + kOffLlrB + (uint32_t)(lane & 15) * 8u;
        const int q0 = max(pcen - 2 * w, 0), q1 = min(pcen + 2 * w, n - 1);
        const int j0 = q0 >> 4, j1 = q1 >> 4;
        for (int jb = j0; jb <= j1; jb += 4) {
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) v[u] = (jb + u <= j1) ? sp[(size_t)(jb + u) * 32] : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (jb + u <= j1) {
                    const int wi = (jb + u - j0) * 4;
                    ring[(wi + 0) * 32] = v[u].x;
                    ring[(wi + 1) * 32] = v[u].y;
                    ring[(wi + 2) * 32] = v[u].z;
                    ring[(wi + 3) * 32] = v[u].w;
                }
            }
        }
        double sc = 0.0, den = 0.0, t2 = 0.0;
        for (int q = q0; q <= q1; q++) {
            const int rel = q - (j0 << 4);
            const uint32_t e = (ring[(rel >> 2) * 32] >> ((rel & 3) * 8)) & 63u;
            const double x = lds_f64(lb + e * 128u);
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
}

__global__ void __launch_bounds__(kV2MaxThreads, 1) k_score_summary_v2(V2Args g)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + kV2AlignSlack - 1) & ~(kV2AlignSlack - 1);
    unsigned char* sm = smem_raw + (sbase - raw);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const DeviceTables* T = g.tabs;
    {
        double2* lut2 = reinterpret_cast<double2*>(sm + kOffLut2);
        for (int i = tid; i <= PLAAC_LUT_LEN; i += blockDim.x) {
            const double l0 = i < PLAAC_LUT_LEN ? T->lut[i] : 0.0;
            const double l1 = i + 1 < PLAAC_LUT_LEN ? T->lut[i + 1] : 0.0;
            lut2[i] = make_double2(l0, l1);
        }
        double2* le = reinterpret_cast<double2*>(sm + kOffLeA);
        for (int i = tid; i < 32 * 8; i += blockDim.x) le[i] = make_double2(T->le0[i >> 3], T->le1[i >> 3]);
        double* la = reinterpret_cast<double*>(sm + kOffLlrA);
        for (int i = tid; i < 32 * 16; i += blockDim.x) la[i] = T->llr[i >> 4];
        double* hy = reinterpret_cast<double*>(sm + kOffHydB);
        double* pa = reinterpret_cast<double*>(sm + kOffPapB);
        double* lb = reinterpret_cast<double*>(sm + kOffLlrB);
        double* hx = reinterpret_cast<double*>(sm + kOffHydX);
        for (int i = tid; i < kTabN * 16; i += blockDim.x) {
            hx[i] = T->hyd[i >> 4];
            hy[i] = T->hydw[i >> 4];
            pa[i] = T->pap[i >> 4];
            lb[i] = T->llr[i >> 4];
        }
    }
    uint32_t* ring_all = reinterpret_cast<uint32_t*>(sm + kV2FixedBytes);
    uint32_t* ring = ring_all + (size_t)wid * g.ring_words * 32 + lane;
    constexpr uint32_t kPadW = 0x01010101u * kPad;
    __syncthreads();

    // Persistent warps: work item = (bucket, role), handed out by one global counter in bucket order (longest
    // buckets first, roles alternating), so every SM keeps all its warps busy with a balanced A/B mix until the
    // queue is empty.  The first round is assigned statically to save one atomic round trip.
    // A warp keeps ONE role while that role has buckets left (odd warps: role B), so the two warps a scheduler
    // partition alternates between mostly run the same loop and the instruction caches hold one role per partition
    // pair; each role has its own bucket counter and a warp whose role has run dry steals from the other one.
    const int64_t nb = g.bv.nbuckets;
    int role = wid & 1;
    const int64_t per_role = (int64_t)(blockDim.x >> 6);
    int64_t item = (int64_t)blockIdx.x * per_role + (wid >> 1);
    const int64_t first_dynamic = (int64_t)gridDim.x * per_role;
    int switched = 0;
    while (true) {
        if (item >= nb) {
            if (switched) break;
            switched = 1;
            role ^= 1;
        } else {
            for (int i = 0; i < g.ring_words; i++) ring[i * 32] = kPadW;
            if (role)
                role_b(g, sbase, ring, lane, item);
            else
                role_a(g, sbase, ring, lane, item);
        }
        unsigned long long nx = 0;
        if (lane == 0) nx = atomicAdd(g.work_counter + role, 1ull);
        item = first_dynamic + (int64_t)__shfl_sync(0xffffffffu, nx, 0);
    }
}

// ------------------------------------------------------------------------------------------------ CORE search
// The -1e6-masked window search of plaac.java:816-833 (hss2 :1206-1257 in reference order: the masking
// constant pollutes the sequential prefix sums, and the jar's COREscore/COREstart carry that pollution),
// then the PrD expansion and PRDscore :851-873.  One lane per listed protein (about 5 % of all).
__global__ void __launch_bounds__(128)
k_core_search(BatchView bv, KScalars ks, const DeviceTables* __restrict__ tabs, plaac_summary* __restrict__ out,
              const int32_t* __restrict__ core_list, const int32_t* __restrict__ core_count)
{
    __shared__ double llr_s[32][16];
    for (int i = threadIdx.x; i < 32 * 16; i += blockDim.x) llr_s[i >> 4][i & 15] = tabs->llr[i >> 4];
    __syncthreads();
    const int total = *core_count;
    const int c = ks.core_len;
    const double big_neg = ks.big_neg;
    const double* lt = &llr_s[0][threadIdx.x & 15];
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int32_t rank = core_list[2 * idx];
        const int64_t b = rank >> 5;
        const int lane = rank & 31;
        const int32_t prot = bv.order[rank];
        const int n = (int)(bv.offsets[prot + 1] - bv.offsets[prot]);
        const int64_t cb = bv.chunk_base[b];
        const uint8_t* sb = reinterpret_cast<const uint8_t*>(bv.stream + cb * 32 + lane);
        const uint32_t* vw = bv.tbw + cb * 32 + lane;
        auto code_at = [&](int i) -> int { return sb[(size_t)(i >> 4) * 512 + (i & 15)] & 31; };
        auto vit_at = [&](int i) -> int { return (vw[(size_t)(i >> 4) * 32] >> (i & 15)) & 1; };
        double ps = 0.0, psl = 0.0, best = 0.0;
        int bstop = c - 1;
        // lead and lag cursors walk their own 16-residue slots
        uint4 lead = make_uint4(0, 0, 0, 0), lag = lead;
        uint32_t vlead = 0, vlag = 0;
        for (int i = 0; i < n; i++) {
            if ((i & 15) == 0) {
                lead = *reinterpret_cast<const uint4*>(sb + (size_t)(i >> 4) * 512);
                vlead = vw[(size_t)(i >> 4) * 32];
            }
            const int k = i - c;
            if (k >= 0 && ((k & 15) == 0 || i == c)) {
                lag = *reinterpret_cast<const uint4*>(sb + (size_t)(k >> 4) * 512);
                vlag = vw[(size_t)(k >> 4) * 32];
            }
            const uint32_t lw = ((i & 12) == 0) ? lead.x : ((i & 12) == 4) ? lead.y : ((i & 12) == 8) ? lead.z : lead.w;
            const int code = (lw >> ((i & 3) * 8)) & 31;
            const double x = ((vlead >> (i & 15)) & 1) ? lt[code * 16] : big_neg;
            ps = ps + x;
            if (k >= 0) {
                const uint32_t gw = ((k & 12) == 0) ? lag.x : ((k & 12) == 4) ? lag.y : ((k & 12) == 8) ? lag.z : lag.w;
                const int codel = (gw >> ((k & 3) * 8)) & 31;
                const double xl = ((vlag >> (k & 15)) & 1) ? lt[codel * 16] : big_neg;
                psl = psl + xl;
                const double d = ps - psl;
                if (d > best) {
                    best = d;
                    bstop = i;
                }
            } else if (i == c - 1) {
                best = ps;
            }
        }
        if (best > big_neg / 2) {
            const int s = bstop - c + 1, e = bstop;
            int a0 = s, a1 = e;
            while (a0 >= 0 && vit_at(a0) == 1) a0--;
            a0++;
            while (a1 < n && vit_at(a1) == 1) a1++;
            a1--;
            double sc = 0.0;
            for (int kk = a0; kk <= a1; kk++) sc = sc + lt[code_at(kk) * 16];
            plaac_summary* r = out + prot;
            r->core_start = s;
            r->core_end = e;
            r->core_score = best;
            r->prd_start = a0;
            r->prd_end = a1;
            r->prd_score = sc;
        }
    }
}

// k masked residues add the masking constant B to the sequential prefix sum k times (hss2 :1230-1233 on the
// masked sequence of :816-831).  For a negative INTEGER B (checked on the host) one such addition is exact
// whenever the result stays inside the binade of ps: both operands are then multiples of the result's ulp.
// So whole stretches are applied as one exact step and only the additions that cross into the next binade
// (about one per power of two) are done one by one -- bit-identical to the jar's k rounded additions.
__device__ __forceinline__ double masked_jump(double ps, int k, double B)
{
    const double aB = -B;
    while (k > 0) {
        double m = 0.0;
        if (ps < 0.0) {
            const double aps = -ps;
            const int ebits = (__double2hiint(aps) >> 20) & 0x7ff;
            const double lim = __hiloint2double((ebits + 1) << 20, 0);  // next power of two above |ps|
            const double room = lim - aps;                             // exact (same binade)
            m = floor(room / aB);
            if (m * aB > room) m -= 1.0;                               // m * aB is an exact integer product
        }
        if (m >= 1.0) {
            const double mm = fmin(m, (double)k);
            ps = ps - mm * aB;  // exact
            k -= (int)mm;
        } else {
            ps = ps + B;  // the rounded addition, as the reference does it
            k -= 1;
        }
    }
    return ps;
}

// Same search as k_core_search with the masked stretches jumped (needs big_neg to be a negative integer).
// Only windows inside Viterbi runs can win (every other window is below big_neg/2 and a listed protein has a run
// of at least c residues), so d = psum[i+1] - psum[i-c+1] is evaluated there only; the lagged prefix sum restarts
// from the lead value at each run start and replays the same additions, so it has the jar's bits.
__global__ void __launch_bounds__(128)
k_core_search_jump(BatchView bv, KScalars ks, const DeviceTables* __restrict__ tabs, plaac_summary* __restrict__ out,
                   const int32_t* __restrict__ core_list, const int32_t* __restrict__ core_count)
{
    __shared__ double llr_s[32][16];
    for (int i = threadIdx.x; i < 32 * 16; i += blockDim.x) llr_s[i >> 4][i & 15] = tabs->llr[i >> 4];
    __syncthreads();
    const int total = *core_count;
    const int c = ks.core_len;
    const double big_neg = ks.big_neg;
    const double* lt = &llr_s[0][threadIdx.x & 15];
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int32_t rank = core_list[2 * idx];
        const uint32_t span = (uint32_t)core_list[2 * idx + 1];
        const int64_t b = rank >> 5;
        const int lane = rank & 31;
        const int32_t prot = bv.order[rank];
        const int n = (int)(bv.offsets[prot + 1] - bv.offsets[prot]);
        const int64_t cb = bv.chunk_base[b];
        const uint8_t* sb = reinterpret_cast<const uint8_t*>(bv.stream + cb * 32 + lane);
        const uint32_t* vw = bv.tbw + cb * 32 + lane;
        auto code_at = [&](int i) -> int { return sb[(size_t)(i >> 4) * 512 + (i & 15)] & 31; };
        // One loop iteration = one Viterbi-1 residue (or one step to the next 16-residue word); masked residues
        // cost nothing: the gap before a residue is applied as one jump.  PRDscore (:870-872, a sequential sum
        // from the run start) and the PrD bounds (:861-866, the enclosing run) are carried along per run.
        double ps = 0.0, lag = 0.0, best = -INFINITY, runsum = 0.0, prd_sc = 0.0;
        int bstop = -1, run = 0, last = 0, run_start = 0, prd_s = -1, prd_e = -2;
        bool hit = false;
        const int nslots = min((n + 15) >> 4, (int)(span >> 16) + 1);  // nothing but masked residues beyond
        int j = (int)(span & 0xffffu) - 1;                              // ... and before (one jump from residue 0)
        uint32_t bits = 0, vnext = vw[(size_t)(j + 1) * 32];
        uint4 cw = make_uint4(0, 0, 0, 0);
        while (true) {
            if (bits == 0) {
                if (++j >= nslots) break;
                const int nb = min(16, n - 16 * j);
                bits = vnext & ((1u << nb) - 1u);
                if (j + 1 < nslots) vnext = vw[(size_t)(j + 1) * 32];
                if (bits) cw = *reinterpret_cast<const uint4*>(sb + (size_t)j * 512);
                continue;
            }
            const int i = __ffs((int)bits) - 1;
            bits &= bits - 1;
            const int p = 16 * j + i;
            if (p != last) {  // masked residues since the previous Viterbi-1 residue: the run (if any) ended
                if (hit) {
                    prd_s = run_start;
                    prd_e = last - 1;
                    prd_sc = runsum;
                    hit = false;
                }
                ps = masked_jump(ps, p - last, big_neg);
                run = 0;
            }
            if (run == 0) {
                lag = ps;
                run_start = p;
                runsum = 0.0;
            }
            const uint32_t w = ((i & 12) == 0) ? cw.x : ((i & 12) == 4) ? cw.y : ((i & 12) == 8) ? cw.z : cw.w;
            const double x = lt[((w >> ((i & 3) * 8)) & 31) * 16];
            ps = ps + x;
            runsum = runsum + x;
            if (run >= c - 1) {
                const double d = ps - lag;
                if (d > best) {
                    best = d;
                    bstop = p;
                    hit = true;
                }
                lag = lag + lt[code_at(p - c + 1) * 16];
            }
            run++;
            last = p + 1;
        }
        if (hit) {
            prd_s = run_start;
            prd_e = last - 1;
            prd_sc = runsum;
        }
        if (best > big_neg / 2) {
            plaac_summary* r = out + prot;
            r->core_start = bstop - c + 1;
            r->core_end = bstop;
            r->core_score = best;
            r->prd_start = prd_s;
            r->prd_end = prd_e;
            r->prd_score = prd_sc;
        }
    }
}

}  // namespace plaac
