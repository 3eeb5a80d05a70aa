// Summary-mode scoring, throughput version "v3": the v2 kernel (summary_kernel_v2.cuh: one lane = one protein, one warp =
// one length bucket, role A = the serial recurrences in reference operation order, role B = the sliding windows as exact
// running sums; same shared-memory layout, same arithmetic, same bits in every column) with fewer issue slots per residue:
//
//   * the Q/N window of the MW column (plaac.java:764-771) is counted four residues at a time in packed bytes (SWAR):
//     flags, the window count after each residue and the "new maximum?" test for a whole word cost ~20 instructions
//     instead of ~12 per residue; only a lane that does see a new maximum walks its four residues one by one;
//   * role B gets (2w+1)^2, cc2 * (2w+1)^2 and cc2 * (2w+1) as doubles from the host instead of re-converting them;
//   * kV3IntFold: role B's hydropathy window sums and the FoldIndex / PAPA sign tests built on them run on the integer
//     pipes (3 IADD3 for the sums, 2 IMAD + ISETP per test, 32-bit table loads) instead of 18 FP64 instructions per
//     residue, where the host proved that the integer sign is v2's FP64 sign (plan_int_fold, plaac_cuda.cu).
//
// OPT is a compile-time bit set; setup_scalars (plaac_cuda.cu) clears each bit whose precondition the parameters do not
// meet.  Measured and dropped (round 2, profiles/r02_kernel_experiments.md): a merged {le0, le1, llr} table entry
// (32-byte stride: two of the eight lanes of a quarter warp always share a bank group, +10 %), the charge window sums on
// the FP64 pipe from a table (three more shared-memory loads per residue, +3 %), a segmented word loop (a second copy of
// the generic body pushes the executed code past the 32 KB instruction cache, +5 %), traceback bits collected per word
// in a nibble (no gain).
#pragma once
#include <type_traits>

#include "common.cuh"
#include "summary_kernel_v2.cuh"

namespace plaac {

constexpr int kV3SwarMw = 1;    // SWAR Q/N window in role A's fast path (needs mw_window <= 100 and the Q/N code set {12, 14})
constexpr int kV3IntFold = 16;  // role B's hydropathy sums and FoldIndex / PAPA sign tests in exact int32 (plan_int_fold)

// (shared-memory layout: v2's, kOff* / kV2FixedBytes / kV2AlignSlack; under kV3IntFold the kOffHydB slots hold
// DeviceTables::hydi in their low word instead of hydw)

__device__ __forceinline__ int lds_s32(uint32_t addr)
{
    int v;
    asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// a*x + b*y + c in wrapping 32-bit arithmetic: the host proved that the true value of every test lies in int32
__device__ __forceinline__ int fold_int(int a, int x, int b, int y, int c)
{
    return (int)((uint32_t)a * (uint32_t)x + (uint32_t)b * (uint32_t)y + (uint32_t)c);
}

// ------------------------------------------------------------------------------------------------ role A
template <int OPT>
__device__ __forceinline__ void role_a3(const V2Args& g, uint32_t sbase, uint32_t* ring, int lane, int64_t b)
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
    uint32_t mwb1 = 0x80808080u;  // SWAR: (min(mw_best, 127) + 1) in every byte
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
        if (!(FAST && (OPT & kV3SwarMw)))
            qn += (int)((ks.qn_mask >> ((w0 >> (8 * i)) & 31u)) & 1u) - (int)((ks.qn_mask >> ((wm >> (8 * i)) & 31u)) & 1u);
        bool tb0 = false, tb1 = false;
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
                tb0 = v10 > v00;
                tb1 = v11 > v01;
                s0 = (tb0 ? v10 : v00) + le.x;
                s1 = (tb1 ? v11 : v01) + le.y;
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
            if (!(FAST && (OPT & kV3SwarMw))) {
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
        }
        acc0 = __funnelshift_r(acc0, tb0 ? 1u : 0u, 1);  // after 16 steps the bit of residue 16j+i sits at 16+i
        acc1 = __funnelshift_r(acc1, tb1 ? 1u : 0u, 1);
    };

    // one word = 4 residues: ring traffic, the three byte streams, 4 steps, traceback word every fourth word
    auto word = [&](auto fast_tag, int wv) {
        constexpr bool FASTW = decltype(fast_tag)::value;
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
        if (FASTW) {
            if (OPT & kV3SwarMw) {
                // Q/N window four residues at a time.  A byte is Q or N iff (code & 0x1d) == 0x0c (codes 14, 12;
                // the pad code 22 and the flag bits 7:5 of the ext byte drop out).  z: bit 7 of a byte = NOT Q/N.
                const uint32_t z0 = (((w0 & 0x1d1d1d1du) ^ 0x0c0c0c0cu) + 0x7f7f7f7fu) >> 7;
                const uint32_t zm = (((wm & 0x1d1d1d1du) ^ 0x0c0c0c0cu) + 0x7f7f7f7fu) >> 7;
                // per byte 1 + isqn(entering) - isqn(leaving), in {0, 1, 2}; multiplying by 0x01010101 gives the
                // inclusive prefix sums of the four bytes (<= 8: no carry between bytes)
                const uint32_t D = (0x01010101u + (zm & 0x01010101u)) - (z0 & 0x01010101u);
                const uint32_t P = D * 0x01010101u;
                // window count after residue i in byte i: counts are >= 0 and <= mw <= 100, so no byte borrows
                const uint32_t Q = ((uint32_t)qn * 0x01010101u + P) - 0x04030201u;
                qn = (int)(Q >> 24);
                // bit 7 of byte i: count_i > mw_best  (mwb1 = mw_best + 1 per byte, 128 while no window is complete)
                if ((((Q | 0x80808080u) - mwb1) & 0x80808080u) != 0u) {
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int q = (int)((Q >> (8 * i)) & 0xffu);
                        if (q > mw_best) {
                            mw_best = q;
                            mw_stop = tbase + i;
                        }
                    }
                    mwb1 = (uint32_t)(mw_best + 1) * 0x01010101u;
                }
            }
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
            if (OPT & kV3SwarMw) mwb1 = (uint32_t)(min(mw_best, 127) + 1) * 0x01010101u;
        }
        if ((wv & 3) == 3) {
            // low half: predecessor-of-state-0 bits of the slot's 16 residues, high half: predecessor-of-state-1 bits
            tbp[(size_t)(wv >> 2) * 32] = __byte_perm(acc0, acc1, 0x7632);
        }
    };

    // fast words: wv != 0, not the word of the first complete LLR / MW window, and tbase + 3 < nmin - 1 (t = nmin-1 stays
    // generic so the "whole protein is one MW window" case, n < mw, is seen there)
    const int fast_end = nmin >= 5 ? (nmin - 1) >> 2 : 0;  // words wv < fast_end have 4*wv + 3 < nmin - 1
#pragma unroll 1
    for (int wv = 0; wv < nwords; wv++) {
        if (wv != 0 && wv != wv_c1 && wv != wv_m1 && wv < fast_end)
            word(std::true_type{}, wv);
        else
            word(std::false_type{}, wv);
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
// Returns true, with no record written, when the integer form of a FoldIndex test or PAPA gate that decides something
// is exactly 0 for a lane of the bucket (IFOLD only): the FP64 sign is then rounding, and the caller scores the bucket
// again with the FP64 sums (GH: hydw read from global memory, the shared slots holding hydi).
template <int OPT, bool GH = false>
__device__ __forceinline__ bool role_b3(const V2Args& g, uint32_t sbase, uint32_t* ring, int lane, int64_t b)
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
    constexpr bool IFOLD = (OPT & kV3IntFold) != 0;

    const uint32_t hb = sbase + kOffHydB + (uint32_t)(lane & 15) * 8u;

    int nmax = n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, d));
    const int t_end = nmax + w;
    const int nwords = (t_end + 3) >> 2;

    double sh = 0;
    int csum = 0;
    double SLh = 0, SGh = 0, Th = 0, Dp = 0, Tp = 0;
    int SLi = 0, SGi = 0, Ti = 0;  // IFOLD: the same window sums in units of 1/q (DeviceTables::hydi)
    int SLc = 0, SGc = 0, Tac = 0;
    double Tb = 0, Wb = 1, vfib = 0;
    int Tacb = 0;      // IFOLD: Tac at the PAPA centre (vfib is rebuilt from it after the loop)
    bool amb = false;  // IFOLD: an integer test that decides something was exactly 0
    int pcen = -1;
    int halfw = ks.h_fi;
    if (halfw > n / 2) halfw = n / 2;
    const int fi_hi = n - halfw;     // FoldIndex scan is over p in [halfw, fi_hi)
    const int edge_hi = n - 1 - w;   // windows centred beyond this are clipped on the right
    int fi_run = 0, fi_numaa = 0, fi_maxrun = 0;  // fi_run: length of the open run of fi < 0 (snaps included)
    uint32_t lo1 = kPadW, lo2 = kPadW;
    const double* hydw = g.tabs->hydw;
    // (host-computed: (double)(2w+1)^2, cc2 * that, cc2 * (2w+1); the compiler otherwise rematerialises the conversion
    // inside the loop to save registers)
    const double WfullD = g.ks_wfull, cc2W = g.ks_cc2w, cc2full = g.ks_cc2full;
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
        // (under IFOLD the FP64 hydropathy loads and conversions below are dead and compiled out)
        const double hy0 = IFOLD ? 0.0 : GH ? hydw[k0 >> 7] : lds_f64(hb | k0), pa0 = lds_f64_off<kOffPapB>(hb | k0);
        const double hy1 = IFOLD ? 0.0 : GH ? hydw[k1 >> 7] : lds_f64(hb | k1), pa1 = lds_f64_off<kOffPapB>(hb | k1);
        const double hy2 = IFOLD ? 0.0 : GH ? hydw[k2 >> 7] : lds_f64(hb | k2), pa2 = lds_f64_off<kOffPapB>(hb | k2);
        const int ch0 = (int)(w0 << (24 - 8 * i)) >> 30;
        const int ch1 = (int)(w1 << (24 - 8 * i)) >> 30;
        const int ch2 = (int)(w2 << (24 - 8 * i)) >> 30;
        if (FAST || t < n) csum += ch0;
        SLc += ch0 - ch1;
        SGc += ch1 - ch2;
        const int aSL = abs(SLc);
        Tac += aSL - abs(SGc);
        const double aSLd = u2d((uint32_t)aSL);
        if (FAST || t < n) sh = sh + lds_f64_off<kOffHydX>(hb | k0);  // mean() :1584, sequential, exact table values
        // window sums of the zero-padded sequence: lead centre p = t-w, lag centre p-(2w+1)
        if (IFOLD) {
            const int h0 = lds_s32(hb | k0), h1 = lds_s32(hb | k1), h2 = lds_s32(hb | k2);
            SLi += h0 - h1;
            SGi += h1 - h2;
            Ti += SLi - SGi;
        } else {
            SLh = (SLh + hy0) - hy1;
            SGh = (SGh + hy1) - hy2;
            Th = (Th + SLh) - SGh;
        }
        Dp = Dp + ((pa0 + pa2) - (pa1 + pa1));  // exact: PAPA log-odds live on a 2^-k grid
        Tp = Tp + Dp;
        const double TacD = u2d((uint32_t)Tac);
        const int p = t - w;
        // IFOLD: a nonzero integer form has the FP64 sign (plan_int_fold); a zero one sets amb
        // FoldIndex run scan :5010-5059 over i in [halfw, n-halfw):
        // sign of fi[p] = cc0*hydro + cc1*|charge| + cc2, scaled by the tap count (> 0)
        if (FAST) {
            // (IFOLD: the host proved that the unclipped integer test is never 0)
            const double fis = IFOLD ? 0.0 : (cc0 * SLh + cc1 * aSLd) + cc2full;
            const bool neg = IFOLD ? fold_int(g.fi_a, SLi, g.fi_b, aSL, g.fi_cfull) < 0 : fis < 0;
            const int closed = (!neg && fi_run >= 5) ? fi_run : 0;
            fi_numaa += closed;
            fi_maxrun = max(fi_maxrun, closed);
            fi_run = neg ? fi_run + 1 : 0;
        } else if (p >= halfw && p < fi_hi) {
            double c2 = cc2full;
            const int taps = full - max(0, w - p) - max(0, p - edge_hi);
            if (p < w || p > edge_hi) c2 = ks.cc2 * u2d((uint32_t)taps);
            const double fis = IFOLD ? 0.0 : (cc0 * SLh + cc1 * aSLd) + c2;
            const int v = IFOLD ? fold_int(g.fi_a, SLi, g.fi_b, aSL, g.fi_c * taps) : 0;
            if (IFOLD && v == 0) amb = true;
            const bool neg = IFOLD ? v < 0 : fis < 0;
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
        // (IFOLD: vfib is not carried; the gate's value at the centre is rebuilt after the loop from Tacb)
        if (FAST) {
            const double vfi = IFOLD ? 0.0 : (cc0 * Th + cc1 * TacD) + cc2W;
            const int v = IFOLD ? fold_int(g.fi_a, Ti, g.fi_b, Tac, g.fi_cw) : 0;
            const bool better = pcen < 0 || Tp * Wb > Tb * WfullD;
            if (IFOLD && better && v == 0) amb = true;
            if (better && (IFOLD ? v < 0 : vfi < 0)) {
                Tb = Tp;
                Wb = WfullD;
                vfib = vfi;
                Tacb = Tac;
                pcen = t - 2 * w;
            }
        } else {
            const int k = p - w;
            if (k >= w && k <= edge_hi) {
                int Wi = Wfull;
                double Wd = WfullD;
                if (k < 2 * w || k > edge_hi - w) {
                    const int ml = 2 * w - k, mr = k - (edge_hi - w);
                    Wi = Wfull - (ml > 0 ? (ml * (ml + 1)) >> 1 : 0) - (mr > 0 ? (mr * (mr + 1)) >> 1 : 0);
                    Wd = u2d((uint32_t)Wi);
                }
                const double vfi = IFOLD ? 0.0 : (cc0 * Th + cc1 * TacD) + ks.cc2 * Wd;
                const int v = IFOLD ? fold_int(g.fi_a, Ti, g.fi_b, Tac, g.fi_c * Wi) : 0;
                const bool better = pcen < 0 || Tp * Wb > Tb * Wd;
                if (IFOLD && better && v == 0) amb = true;
                if (better && (IFOLD ? v < 0 : vfi < 0)) {
                    Tb = Tp;
                    Wb = Wd;
                    vfib = vfi;
                    Tacb = Tac;
                    pcen = k;
                }
            }
        }
    };

    uint4 nxt = make_uint4(kPadW, kPadW, kPadW, kPadW);
    if (nch > 0) nxt = sp[0];
    auto word = [&](auto fast_tag, int wv) {
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
#pragma unroll
        for (int i = 0; i < 4; i++) step(fast_tag, tbase + i, i, w0, w1, w2);
    };
    // fast words: tbase >= 4w and tbase + 3 < nmin - 1 (t <= nmin-2 keeps the last scanned FoldIndex position,
    // p = n-1-halfw, out of the fast path)
    const int fast_end = nmin >= 5 ? (nmin - 1) >> 2 : 0;
    const int fast_begin = (fast_lo + 3) >> 2;
#pragma unroll 1
    for (int wv = 0; wv < nwords; wv++) {
        if (wv >= fast_begin && wv < fast_end)
            word(std::true_type{}, wv);
        else
            word(std::false_type{}, wv);
    }

    if (IFOLD && __any_sync(0xffffffffu, amb)) return true;
    if (prot < 0) return false;
    plaac_summary* r = g.out + prot;
    if (n < 1) {
        r->fi_numaa = r->fi_maxrun = r->papa_center = 0;
        r->fi_meanhydro = r->fi_meancharge = r->fi_meancombo = 0;
        r->papa_combo = r->papa_prop = r->papa_fi = r->papa_llr = r->papa_llr2 = 0;
        return false;
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
        if (!IFOLD) r->papa_fi = vfib / Wb;
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
        double sc = 0.0, den = 0.0, t2 = 0.0, th = 0.0;
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
            // IFOLD: v2's Th at the centre; the products and sums on the hydw grid are exact, so any order gives its bits
            if (IFOLD) th = th + hydw[e] * (double)(full - dist);
        }
        // the PAPA gate's FP64 value at the centre; cc2 * Wb is the product v2 added (the host's cc2W: the same)
        if (IFOLD) r->papa_fi = ((cc0 * th + cc1 * u2d((uint32_t)Tacb)) + ks.cc2 * Wb) / Wb;
        r->papa_llr = sc / den;
        r->papa_llr2 = t2 / Wb;
    } else {
        r->papa_combo = -INFINITY;
        r->papa_prop = r->papa_fi = r->papa_llr = r->papa_llr2 = nan("");
    }
    return false;
}

// 768 threads (kV2MaxThreads): 80 registers per thread
template <int OPT>
__global__ void __launch_bounds__(kV2MaxThreads, 1) k_score_summary_v3(V2Args g)
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
            if (OPT & kV3IntFold)
                reinterpret_cast<int2*>(hy)[i] = make_int2(T->hydi[i >> 4], 0);
            else
                hy[i] = T->hydw[i >> 4];
            pa[i] = T->pap[i >> 4];
            lb[i] = T->llr[i >> 4];
        }
    }
    uint32_t* ring_all = reinterpret_cast<uint32_t*>(sm + kV2FixedBytes);
    uint32_t* ring = ring_all + (size_t)wid * g.ring_words * 32 + lane;
    constexpr uint32_t kPadW = 0x01010101u * kPad;
    __syncthreads();

    // Persistent warps, one role per warp while that role has buckets left (see k_score_summary_v2), both roles on every
    // scheduler partition (measured 1 % faster than one role per partition, round 2): warps 2k and 2k+1 take different
    // roles, and the roles alternate along every partition (wid & 3).
    const int64_t nb = g.bv.nbuckets;
    int role = ((wid >> 2) ^ wid) & 1;
    const int64_t per_role = (int64_t)(blockDim.x >> 6);
    const int slot_in_role = wid >> 1;
    int64_t item = (int64_t)blockIdx.x * per_role + slot_in_role;
    const int64_t first_dynamic = (int64_t)gridDim.x * per_role;
    int switched = 0;
    while (true) {
        if (item >= nb) {
            if (switched) break;
            switched = 1;
            role ^= 1;
        } else {
            for (int i = 0; i < g.ring_words; i++) ring[i * 32] = kPadW;
            if (role) {
                if (role_b3<OPT>(g, sbase, ring, lane, item)) {
                    for (int i = 0; i < g.ring_words; i++) ring[i * 32] = kPadW;
                    role_b3<OPT & ~kV3IntFold, true>(g, sbase, ring, lane, item);
                }
            } else {
                role_a3<OPT>(g, sbase, ring, lane, item);
            }
        }
        unsigned long long nx = 0;
        if (lane == 0) nx = atomicAdd(g.work_counter + role, 1ull);
        item = first_dynamic + (int64_t)__shfl_sync(0xffffffffu, nx, 0);
    }
}

// Every subset of the default bits has an instantiation: setup_scalars clears bits per parameter set.
constexpr int kV3DefaultOpt = kV3SwarMw | kV3IntFold;
using V3Kernel = void (*)(V2Args);
inline V3Kernel v3_kernel(int opt)
{
    switch (opt) {
        case 0: return k_score_summary_v3<0>;
        case kV3SwarMw: return k_score_summary_v3<kV3SwarMw>;
        case kV3IntFold: return k_score_summary_v3<kV3IntFold>;
        case kV3SwarMw | kV3IntFold: return k_score_summary_v3<kV3SwarMw | kV3IntFold>;
    }
    return nullptr;
}

}  // namespace plaac
