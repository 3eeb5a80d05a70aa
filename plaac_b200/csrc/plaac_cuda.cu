// libplaac_cuda.so -- C ABI (include/plaac_cuda.h) over the sm_100a kernels.
// No CPU fallback: every entry point either runs the CUDA path or returns an error code.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "prep.cuh"
#include "ingest.cuh"
#include "rank.cuh"
#include "residue_kernel.cuh"
#include "residue_kernel_v2.cuh"
#include "summary_kernel.cuh"
#include "summary_kernel_v2.cuh"
#include "summary_kernel_v3.cuh"
#include "long_kernel.cuh"
#include "long_residue.cuh"
#include "lean.cuh"
#include "generic_windows.cuh"
#include "variants.cuh"
#include "segments.cuh"
#include "shuffle.cuh"
#include "shuffle_seq.cuh"

using namespace plaac;

namespace {

thread_local std::string g_last_error = "";

// Integer form of the v3 kernel's FoldIndex / PAPA sign tests (kV3IntFold, plan_int_fold): hydw[c] ~ h[c] / q and
// M * (cc0 * X + cc1 * C + cc2 * taps) = a * (sum of h) + b * C + c * taps
struct IntFold {
    int32_t h[PLAAC_NAA];
    int32_t a, b, c;
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// One set of device work buffers; plaac_score() cycles through kSlots of them to overlap copies with compute.
struct Slot {
    cudaStream_t stream = nullptr;
    DevBuf hist, cursor, order, nchunks, chunk_base, stream_buf, tbw, slot_bucket, errflag, core_list, core_count, scan_tmp, gen_f64;
    DevBuf codes, offsets, summaries;  // staging for the host-buffer API
    DevBuf words, lengths;             // ... of its packed form (plaac_score_packed)
    DevBuf v_prot, v_first, v_pos, v_code;  // the chunk's slice of a variant list (plaac_score_variants)
    DevBuf v_effects;                       // the chunk's effects (plaac_score_variant_effects) or null values
    DevBuf sh_rep;                          // the chunk's replicates (plaac_score_shuffles): ShuffleRep each
    DevBuf sg_cnt, sg_first, sg_ent;        // the chunk's segments (plaac_score_segments): counts, their scan, entries
    DevBuf hit_flag, hit_pos;          // compact ranked output (plaac_hits)
    DevBuf res_u8, res_f64;            // per-residue staging for the host-buffer API
    DevBuf res_b0, res_b1, res_a0, res_a1, res_mapw, res_lpseq;  // per-residue scratch (bucketed layout)
    DevBuf ing_agg, ing_cnt, ing_base, ing_misc;                 // FASTA ingest scratch
    DevBuf ing_text, ing_codes, ing_offsets, ing_npos, ing_nlen, ing_flags, ing_hist;  // staging for the host-buffer ingest
    DevBuf rk_keys[2], rk_vals[2], rk_hist, rk_offs, rk_order;                         // ranking scratch
    DevBuf lg_list, lg_off, lg_cnt, lg_ext, lg_ext_win, lg_tb, lg_vit;                          // long-sequence path
    DevBuf lp_s0, lp_s1, lp_bnd, lp_lpseq;          // ... in per-residue mode (long_residue.cuh)
    DevBuf lg_hmm, lg_sum0, lg_vb;                  // ... records with the HMM columns from k_long_post (k_long_final)
    unsigned long long* h_long = nullptr;  // pinned: [0] long proteins, [1] scratch residues, or 3 x kLongBins bins
    DevBuf lg_bins;
    cudaStream_t aux1 = nullptr, aux2 = nullptr, aux3 = nullptr, aux4 = nullptr, aux5 = nullptr;
    // staging for callers whose buffers are pageable (plaac_score): pinned copies of the chunk's codes and records
    void* h_stage_codes = nullptr;
    size_t h_stage_codes_cap = 0;
    void* h_stage_sum = nullptr;
    size_t h_stage_sum_cap = 0;
    void* out_dst = nullptr;  // where the staged records (or effects) of the chunk in flight go once it has finished
    size_t out_bytes = 0;
    cudaEvent_t ev_fork = nullptr, ev_j1 = nullptr, ev_j2 = nullptr, ev_j3 = nullptr, ev_j4 = nullptr, ev_j5 = nullptr;
    // segments of the chunk in flight (plaac_score_segments): pinned copies of its first[] and of its stored entries,
    // and what a rerun of the bounds / score kernels needs if the entries overflowed seg_cap
    void* h_sg_first = nullptr;
    size_t h_sg_first_cap = 0;
    void* h_sg_ent = nullptr;
    size_t h_sg_ent_cap = 0;
    SegArgs seg_args;
    int64_t seg_np = -1, seg_cap = 0, seg_p0 = 0;  // proteins of the chunk (-1: no segments pending), capacity, first protein
    int64_t* h_total = nullptr;        // pinned
    int* h_err = nullptr;              // pinned
    cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_c = nullptr, ev_d = nullptr;
    bool timing_valid = false;
};

}  // namespace

// plaac_score() pipelines its chunks over this many sets of device buffers: chunk i+1's and i+2's host->device copies are
// queued while chunk i computes and copies back, so the copy engine never waits for the host (with two sets it did:
// 0.7 ms per chunk, measured).
constexpr int kSlots = 3;

struct plaac_ctx {
    int device = 0;
    plaac_params params;
    KScalars ks;
    DeviceTables* d_tabs = nullptr;
    Slot slot[kSlots];
    DevBuf all_summaries;      // records of a whole host-buffer call, kept on the device for the compact ranked output
    DevBuf union_rec, union_idx, union_order, union_out_idx;  // plaac_score_multi_packed: the shards' hit rows merged on this GPU
    DevBuf var_ref, var_ref_off;  // reference batch of plaac_score_variants, uploaded once per call
    DevBuf var_wild;              // its records (plaac_score_variant_effects), or the observed records of the selection
                                  // (plaac_score_shuffles), uploaded once per call
    DevBuf null_counts;           // plaac_score_shuffles: nsel x k counts, summed over the chunks
    // plaac_score_shuffles_seq: nsel x k replicates scored (null_counts holds the hits), the round's hit flags, the
    // active flags of its list and their scan, and the list itself (two buffers, [0] = length, then the entries)
    DevBuf seq_scored, seq_flags, seq_live, seq_pos, seq_act[2];
    // pageable <-> device copies of the FASTA calls: two pinned staging buffers, filled / emptied by a multi-threaded memcpy
    void* stage_buf[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    bool stage_pending[2] = {false, false};
    int nwarps = 0, ring_words = 0;
    size_t smem_bytes = 0;
    int v2_nwr = 0;            // warps per role of the v2 and v3 kernels (0 = both unavailable for these params)
    size_t v2_smem_bytes = 0;  // ... and their shared memory (the same layout)
    int v3_opt = 0;            // option bits of the v3 kernel (summary_kernel_v3.cuh)
    IntFold ifold = {};        // valid when v3_opt has kV3IntFold
    int v2_always_in = 0;     // forward recurrence provably keeps |a-b| < 40 (no LUT range test needed)
    ResidueV2Plan res_plan;
    int variant = 0;           // 0 auto, 1 = v1 (reference-order anchor), 2 = v2
    std::string v2_why;
    int sm_count = 0;
    bool generic_windows = false;  // ww1, ww2, ww3 with different half-widths: generic_windows.cuh
    plaac_stats stats;
    int64_t chunk_res = (int64_t)256 << 20, chunk_res_pr = (int64_t)32 << 20, chunk_prot = (int64_t)4 << 20;
    // long-sequence path: > 0 fixed threshold (default 8192), -1 automatic threshold per batch, 0 off.  Both paths give
    // the same bytes for every column, so the choice never shows in the results.
    int64_t long_min = 8192;
    int long_warm = 256;       // forward warm-up of that path
    unsigned long long long_tie[4] = {0, 0, 0, 0};  // binades with an exact rounding tie among the table constants
    int64_t lp_big_min = kLpBigMin;  // proteins of at least this many residues take k_long_post's cluster launch
    std::string err;
    int last_slot = 0;
};

namespace {

int fail(plaac_ctx* ctx, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx)
        ctx->err = buf;
    else
        g_last_error = buf;
    return code;
}

// Function-try-block handler of every extern "C" entry point: nothing may throw across the C ABI (include/plaac_cuda.h).
int api_caught(plaac_ctx* ctx, const char* fn) noexcept
{
    int code = PLAAC_E_INVALID;
    char what[200] = "unknown C++ exception";
    try {
        throw;
    } catch (const std::bad_alloc&) {
        code = PLAAC_E_NOMEM;
        snprintf(what, sizeof(what), "out of host memory");
    } catch (const std::exception& e) {
        snprintf(what, sizeof(what), "%s", e.what());
    } catch (...) {
    }
    try {
        return fail(ctx, code, "%s: %s", fn, what);
    } catch (...) {
        return code;
    }
}

#define CU(ctx, call)                                                                                      \
    do {                                                                                                   \
        cudaError_t e__ = (call);                                                                          \
        if (e__ != cudaSuccess)                                                                            \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? PLAAC_E_NOMEM : PLAAC_E_CUDA, "%s: %s", #call, \
                        cudaGetErrorString(e__));                                                          \
    } while (0)

int cu_rc(plaac_ctx* ctx, cudaError_t e, const char* what)
{
    if (e == cudaSuccess) return PLAAC_OK;
    return fail(ctx, e == cudaErrorMemoryAllocation ? PLAAC_E_NOMEM : PLAAC_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

int ensure(plaac_ctx* ctx, DevBuf& b, size_t bytes)
{
    if (bytes <= b.cap) return PLAAC_OK;
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 8 + 256;  // a little slack so similar batches do not realloc
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMalloc(&b.p, bytes + 256);
        want = bytes + 256;
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, PLAAC_E_NOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        }
    }
    b.cap = want;
    return PLAAC_OK;
}

void release(DevBuf& b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

int next_pow2(int x)
{
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

bool plan_int_fold(const plaac_params& P, int w, IntFold& f);

int setup_scalars(plaac_ctx* ctx)
{
    const plaac_params& P = ctx->params;
    KScalars& k = ctx->ks;
    if (P.core_len < 1) return fail(ctx, PLAAC_E_INVALID, "core_len must be >= 1 (got %d)", P.core_len);
    if (P.ww1 < 1 || P.ww2 < 1 || P.ww3 < 1) return fail(ctx, PLAAC_E_INVALID, "window sizes must be >= 1");
    if (P.mw_window < 1) return fail(ctx, PLAAC_E_INVALID, "mw_window must be >= 1");
    // The streaming kernels carry one half-width.  Window sizes with different half-widths (-w and -W of the jar are
    // independent) take the tap-by-tap kernels of generic_windows.cuh for everything that depends on the windows; the
    // streaming kernels then run with ww1 for all three (their window columns are overwritten).
    ctx->generic_windows = P.ww1 / 2 != P.ww2 / 2 || P.ww1 / 2 != P.ww3 / 2 || (P.ww1 - 1) / 2 != (P.ww2 - 1) / 2;
    // ... and so do windows whose look-back (4w + 2 residues) would crowd the residue rings out of shared memory; the
    // streaming kernels then run with the default window
    int ww_stream = P.ww1;
    if (4 * (P.ww1 / 2) + 2 > 512) {
        ctx->generic_windows = true;
        ww_stream = 41;
    }
    k.core_len = P.core_len;
    k.w = ww_stream / 2;
    k.h_fi = (ww_stream - 1) / 2;
    k.h_papa = ctx->generic_windows ? (ww_stream - 1) / 2 : (P.ww2 - 1) / 2;
    k.mw_window = P.mw_window;
    k.adjust_prolines = P.adjust_prolines ? 1 : 0;
    k.charge_plus = k.charge_minus = 0;
    for (int i = 0; i < PLAAC_NAA; i++) {
        if (P.charge[i] == 1.0)
            k.charge_plus |= 1u << i;
        else if (P.charge[i] == -1.0)
            k.charge_minus |= 1u << i;
        else if (P.charge[i] != 0.0)
            return fail(ctx, PLAAC_E_UNSUPPORTED, "charge[%d]=%g: only -1, 0, +1 are supported", i, P.charge[i]);
    }
    k.qn_mask = (1u << 12) | (1u << 14);  // N, Q  (qnmask, plaac.java:733)
    k.lt00 = P.lt[0][0];
    k.lt01 = P.lt[0][1];
    k.lt10 = P.lt[1][0];
    k.lt11 = P.lt[1][1];
    k.li0 = P.li[0];
    k.li1 = P.li[1];
    k.lf0 = P.lf[0];
    k.lf1 = P.lf[1];
    k.cc0 = P.fi_cc[0];
    k.cc1 = P.fi_cc[1];
    k.cc2 = P.fi_cc[2];
    k.big_neg = P.big_neg;
    k.ln2 = P.ln2;

    const int maxoff = std::max(std::max(4 * k.w + 2, k.core_len), k.mw_window);
    ctx->ring_words = next_pow2((maxoff + 16 + 3) / 4 + 1);
    const size_t per_warp = (size_t)ctx->ring_words * 32 * sizeof(uint32_t);
    const size_t fixed = sizeof(SummarySmem);
    const size_t limit = 227 * 1024;
    if (fixed + per_warp > limit)
        return fail(ctx, PLAAC_E_UNSUPPORTED, "core_len/window look-back of %d residues does not fit the shared-memory ring",
                    maxoff);
    ctx->nwarps = (int)std::min<size_t>(12, (limit - fixed) / per_warp);
    ctx->smem_bytes = fixed + per_warp * ctx->nwarps;

    // v2 preconditions: loglut[0] == ln2 bit for bit (lets the a == b branch of logeapeb fold into the
    // interpolation) and hmm0's emissions identical to hmm1's background state (as prionhmm0/1 build them).
    ctx->v2_nwr = 0;
    if (memcmp(&P.loglut[0], &P.ln2, sizeof(double)) != 0)
        ctx->v2_why = "loglut[0] != ln2";
    else if (memcmp(P.le0, P.le[0], sizeof(P.le0)) != 0)
        ctx->v2_why = "hmm0 emissions differ from hmm1 state 0";
    else {
        const size_t fixed2 = (size_t)kV2FixedBytes + kV2AlignSlack;
        if (fixed2 + 2 * per_warp <= limit) {
            const int nwr = (int)std::min<size_t>(kV2MaxThreads / 64, (limit - fixed2) / (2 * per_warp));
            ctx->v2_nwr = nwr;
            ctx->v2_smem_bytes = fixed2 + per_warp * 2 * nwr;
        } else
            ctx->v2_why = "ring does not fit beside the v2 tables";
        // v3: same design, warps and shared-memory layout, fewer issue slots per residue (summary_kernel_v3.cuh)
        if (ctx->v2_nwr > 0) {
            int opt = kV3DefaultOpt;
            // the packed Q/N window needs counts that fit a byte and the jar's Q/N code set
            if (P.mw_window > 100 || k.qn_mask != ((1u << 12) | (1u << 14))) opt &= ~kV3SwarMw;
            // ... and the integer FoldIndex tests a proof that they give the FP64 signs for these tables and windows
            if (!plan_int_fold(P, k.w, ctx->ifold)) opt &= ~kV3IntFold;
            ctx->v3_opt = opt;
        }
        // Range of d = a0 - a1 in the forward recurrence: alpha0/alpha1 is a Moebius image of the previous
        // ratio, so for t >= 1  d in [lt10 - lt11 + min(le0-le1), lt00 - lt01 + max(le0-le1)], and the two
        // log-sum-exp arguments differ by (lt0i - lt1i) + d.  If that is safely below 40 the LUT range test
        // (logeapeb's `c < 40`, plaac.java:1027) can never fail and the kernel skips it.
        double dmin = INFINITY, dmax = -INFINITY;
        for (int cidx = 0; cidx < PLAAC_NAA; cidx++) {
            const double dl = P.le[0][cidx] - P.le[1][cidx];
            dmin = std::min(dmin, dl);
            dmax = std::max(dmax, dl);
        }
        const double m1 = P.lt[1][0] - P.lt[1][1], m2 = P.lt[0][0] - P.lt[0][1], m0 = P.li[0] - P.li[1];
        const double lo = std::min(std::min(m1, m2), m0) + dmin;
        const double hi = std::max(std::max(m1, m2), m0) + dmax;
        const double dabs = std::max(std::fabs(lo), std::fabs(hi));
        const double targ = std::max(std::fabs(P.lt[0][0] - P.lt[1][0]), std::fabs(P.lt[0][1] - P.lt[1][1])) + dabs;
        ctx->v2_always_in = (std::isfinite(targ) && targ < 39.0) ? 1 : 0;
    }
    return PLAAC_OK;
}

// The PAPA window sums are running sums (add the entering residue, subtract the leaving one).  To keep
// them drift-free and, above all, to keep EXACT ties exact (PAPAcen is a first-strict-maximum search,
// plaac.java:4941-4948), the PAPA log-odds are rounded to a grid 2^-k coarse enough that every partial sum
// of up to (2w+1)^2 of them is exactly representable: all those double additions are then exact.
// Grid error <= 2^-41 for the default windows (values ~0.1 => ~5e-12 relative).  Not applied when the
// grid would be coarser than 2^-38 (huge windows) or a table entry is not finite.
double sum_grid(const double* tab, int w)
{
    double maxabs = 0;
    for (int c = 0; c < PLAAC_NAA; c++) {
        if (!std::isfinite(tab[c])) return 0.0;
        maxabs = std::max(maxabs, std::fabs(tab[c]));
    }
    if (maxabs == 0) return 0.0;
    const double taps = (2.0 * w + 2.0) * (2.0 * w + 2.0);
    int e = 0;
    std::frexp(taps * maxabs, &e);  // taps*maxabs < 2^e
    const int k = e - 52;          // grid 2^k keeps sums below 2^52 grid units
    if (k > -38) return 0.0;
    return std::ldexp(1.0, k);
}

// hydropathy on the exact-sum grid gridh = sum_grid(P.hydro2, w) (DeviceTables::hydw)
double hyd_on_grid(const plaac_params& P, int c, double gridh)
{
    return gridh > 0 ? std::nearbyint(P.hydro2[c] / gridh) * gridh : P.hydro2[c];
}

// ifold: the integer hydropathy table of kV3IntFold, or null
void fill_tables(const plaac_params& P, DeviceTables& T, int w, const IntFold* ifold)
{
    memset(&T, 0, sizeof(T));
    const double grid = sum_grid(P.papa_lod, w);
    // The hydropathy window sums get the same treatment (grid 2^-41 for PLAAC's tables: 2e-13 relative to a window
    // mean): the summary kernels' FoldIndex columns then do not depend on how a running sum was started, so the
    // bucketed kernel and the chunked long-sequence path give the same bits.
    const double gridh = sum_grid(P.hydro2, w);
    for (int e = 0; e < kTabN; e++) {
        const int c = e & 31;
        if (c >= PLAAC_NAA) continue;  // pad and unused codes: all zero
        T.le0[e] = P.le[0][c];
        T.le1[e] = P.le[1][c];
        T.lebg[e] = P.le0[c];
        T.llr[e] = P.llr[c];
        T.hyd[e] = P.hydro2[c];
        T.hydw[e] = hyd_on_grid(P, c, gridh);
        if (ifold) T.hydi[e] = ifold->h[c];
        double pl = P.papa_lod[c];
        if (grid > 0) pl = std::nearbyint(pl / grid) * grid;
        T.pap[e] = (e & kPapaMaskBit) ? 0.0 : pl;
    }
    for (int i = 0; i < PLAAC_LUT_LEN; i++) T.lut[i] = P.loglut[i];
}

// Smallest d in [1, maxd] with x*d within 1e-9 of an integer n (the tolerance only picks the candidate; plan_int_fold's
// error bound decides), or 0.
int64_t small_denominator(double x, int64_t maxd, int64_t& n)
{
    if (!(std::fabs(x) < 1e6)) return 0;
    for (int64_t d = 1; d <= maxd; d++) {
        const double y = x * (double)d;
        if (std::fabs(y - std::nearbyint(y)) <= 1e-9) {
            n = (int64_t)std::nearbyint(y);
            return d;
        }
    }
    return 0;
}

// Can the v3 kernel's role B test the signs of fi = (cc0 * X + cc1 * C) + cc2 * taps (X = a hydropathy window sum on the
// hydw grid, C = |charge sum|; the FoldIndex run test over 2w+1 taps, the PAPA gate over (2w+1)^2) in exact int32?
//   * the grid must be in use: only then is X exactly the sum of hydw, independent of order;
//   * hydw[c] ~ h[c] / q and cc_i ~ n_i / d_i with small q, d_i, so that for M = lcm(q d0, d1, d2) the rational value
//     of fi is V / M, V = a * sum(h) + b * C + c * taps an integer (PLAAC: q = 90, M = 18000, V = 557 S - 18000 C - 20718 taps);
//   * every V over the (2w+1)^2 taps of the PAPA gate lies in int32 (the kernel wraps, only the final value counts);
//   * the FP64 value v2 computes differs from V / M by at most E (representation errors of the tables and coefficients,
//     five roundings), and E < 1 / (2M): where V != 0, |V / M| >= 1/M and the FP64 value has V's sign.
// A bucket where a deciding test has V == 0 is scored again with the FP64 sums (role_b3).
bool plan_int_fold(const plaac_params& P, int w, IntFold& f)
{
    const double gridh = sum_grid(P.hydro2, w);
    if (!(gridh > 0)) return false;
    double hw[PLAAC_NAA];
    double hmax = 0;
    for (int c = 0; c < PLAAC_NAA; c++) {
        hw[c] = hyd_on_grid(P, c, gridh);
        hmax = std::max(hmax, std::fabs(hw[c]));
    }
    int q = 0;
    for (int qq = 1; qq <= 1000 && q == 0; qq++) {
        bool ok = true;
        for (int c = 0; c < PLAAC_NAA && ok; c++) ok = std::fabs(hw[c] * qq - std::nearbyint(hw[c] * qq)) <= 1e-9;
        if (ok) q = qq;
    }
    if (q == 0) return false;
    int64_t num[3], den[3];
    for (int i = 0; i < 3; i++)
        if ((den[i] = small_denominator(P.fi_cc[i], 10000, num[i])) == 0) return false;
    const int64_t d0 = q * den[0];
    int64_t M = d0 / std::gcd(d0, den[1]) * den[1];
    M = M / std::gcd(M, den[2]) * den[2];
    if (M >= ((int64_t)1 << 31)) return false;
    const double coef[3] = {(double)(num[0] * (M / d0)), (double)(num[1] * (M / den[1])), (double)(num[2] * (M / den[2]))};
    // value range over every window: sum(h) in W*[min(0, hmin), max(0, hmax)] (padding counts 0), C in [0, W], taps in [1, W]
    const double full = 2.0 * w + 1.0, W = full * full;
    double hlo = 0, hhi = 0;
    for (int c = 0; c < PLAAC_NAA; c++) {
        f.h[c] = (int32_t)std::nearbyint(hw[c] * q);
        hlo = std::min(hlo, (double)f.h[c]);
        hhi = std::max(hhi, (double)f.h[c]);
    }
    const double lim = 2147483647.0;
    const double vlo = std::min(coef[0] * hlo * W, coef[0] * hhi * W) + std::min(0.0, coef[1] * W) + std::min(coef[2], coef[2] * W);
    const double vhi = std::max(coef[0] * hlo * W, coef[0] * hhi * W) + std::max(0.0, coef[1] * W) + std::max(coef[2], coef[2] * W);
    if (!(vlo > -lim && vhi < lim && std::max(-hlo, hhi) * W < lim)) return false;
    // error bound at W taps (the larger test); every value below is an upper bound, with one ulp for its own rounding
    constexpr double u = 1.0 / 4503599627370496.0;  // 2^-52
    double eh = 0;  // max |hw[c] - h[c]/q|
    for (int c = 0; c < PLAAC_NAA; c++) eh = std::max(eh, (std::fabs(hw[c] * q - f.h[c]) + u * std::fabs(hw[c] * q)) / q);
    double dc[3];  // |cc_i - n_i/d_i|
    for (int i = 0; i < 3; i++) {
        const double y = P.fi_cc[i] * (double)den[i];
        dc[i] = (std::fabs(y - (double)num[i]) + u * std::fabs(y)) / (double)den[i];
    }
    const double cc0 = std::fabs(P.fi_cc[0]), cc1 = std::fabs(P.fi_cc[1]), cc2 = std::fabs(P.fi_cc[2]);
    const double mag = (cc0 * hmax + cc1 + cc2) * W;  // bound on every intermediate of the FP64 expression
    const double E = (dc[0] * hmax + cc0 * eh + dc[1] + dc[2]) * W + 5.0 * u * mag;
    if (!(E * (double)M < 0.5)) return false;
    // the kernel does not look for zeros of its unclipped FoldIndex test (2w+1 residues, |charge sum| C <= 2w+1): no
    // sum of hydi over 2w+1 residues may give V == 0 there
    for (int64_t C = 0; C <= 2 * w + 1; C++) {
        const int64_t rest = -((int64_t)coef[1] * C + (int64_t)coef[2] * (2 * w + 1));
        if (coef[0] == 0 ? rest == 0 : (rest % (int64_t)coef[0] == 0 && rest / (int64_t)coef[0] >= hlo * full &&
                                        rest / (int64_t)coef[0] <= hhi * full))
            return false;
    }
    f.a = (int32_t)coef[0];
    f.b = (int32_t)coef[1];
    f.c = (int32_t)coef[2];
    return true;
}

int slot_init(plaac_ctx* ctx, Slot& s)
{
    CU(ctx, cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    CU(ctx, cudaMallocHost((void**)&s.h_total, sizeof(int64_t)));
    CU(ctx, cudaMallocHost((void**)&s.h_err, sizeof(int)));
    CU(ctx, cudaMallocHost((void**)&s.h_long, 3 * kLongBins * sizeof(unsigned long long)));
    CU(ctx, cudaEventCreate(&s.ev_a));
    CU(ctx, cudaEventCreate(&s.ev_b));
    CU(ctx, cudaEventCreate(&s.ev_c));
    CU(ctx, cudaEventCreate(&s.ev_d));
    CU(ctx, cudaStreamCreateWithFlags(&s.aux1, cudaStreamNonBlocking));
    CU(ctx, cudaStreamCreateWithFlags(&s.aux2, cudaStreamNonBlocking));
    CU(ctx, cudaStreamCreateWithFlags(&s.aux3, cudaStreamNonBlocking));
    CU(ctx, cudaStreamCreateWithFlags(&s.aux4, cudaStreamNonBlocking));
    CU(ctx, cudaStreamCreateWithFlags(&s.aux5, cudaStreamNonBlocking));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_j1, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_j2, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_j3, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_j4, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_j5, cudaEventDisableTiming));
    int rc = ensure(ctx, s.errflag, sizeof(int));
    if (rc) return rc;
    CU(ctx, cudaMemsetAsync(s.errflag.p, 0, sizeof(int), s.stream));
    if ((rc = ensure(ctx, s.lg_cnt, 32))) return rc;
    CU(ctx, cudaMemsetAsync(s.lg_cnt.p, 0, 32, s.stream));
    return PLAAC_OK;
}

void slot_free(Slot& s)
{
    for (DevBuf* b : {&s.gen_f64, &s.scan_tmp, &s.hist, &s.cursor, &s.order, &s.nchunks, &s.chunk_base, &s.stream_buf, &s.tbw, &s.slot_bucket, &s.errflag,
                      &s.core_list, &s.core_count, &s.codes, &s.offsets, &s.summaries, &s.words, &s.lengths, &s.v_prot, &s.v_first, &s.v_pos, &s.v_code, &s.v_effects, &s.sh_rep, &s.sg_cnt, &s.sg_first, &s.sg_ent, &s.hit_flag, &s.hit_pos, &s.res_u8, &s.res_f64, &s.res_b0,
                      &s.res_b1, &s.res_a0, &s.res_a1, &s.res_mapw, &s.res_lpseq, &s.ing_agg, &s.ing_cnt, &s.ing_base,
                      &s.ing_misc, &s.ing_text, &s.ing_codes, &s.ing_offsets, &s.ing_npos, &s.ing_nlen, &s.ing_flags,
                      &s.ing_hist, &s.rk_keys[0], &s.rk_keys[1], &s.rk_vals[0], &s.rk_vals[1], &s.rk_hist, &s.rk_offs,
                      &s.rk_order, &s.lg_list, &s.lg_off, &s.lg_cnt, &s.lg_ext, &s.lg_ext_win, &s.lg_tb, &s.lg_vit, &s.lg_bins, &s.lp_s0, &s.lp_s1, &s.lp_bnd, &s.lp_lpseq, &s.lg_hmm, &s.lg_sum0, &s.lg_vb})
        release(*b);
    if (s.h_long) cudaFreeHost(s.h_long);
    if (s.h_stage_codes) cudaFreeHost(s.h_stage_codes);
    if (s.h_stage_sum) cudaFreeHost(s.h_stage_sum);
    if (s.h_sg_first) cudaFreeHost(s.h_sg_first);
    if (s.h_sg_ent) cudaFreeHost(s.h_sg_ent);
    s.h_stage_codes = s.h_stage_sum = nullptr;
    s.h_stage_codes_cap = s.h_stage_sum_cap = 0;
    if (s.h_total) cudaFreeHost(s.h_total);
    if (s.h_err) cudaFreeHost(s.h_err);
    for (cudaEvent_t e : {s.ev_a, s.ev_b, s.ev_c, s.ev_d, s.ev_fork, s.ev_j1, s.ev_j2, s.ev_j3, s.ev_j4, s.ev_j5})
        if (e) cudaEventDestroy(e);
    for (cudaStream_t a : {s.aux1, s.aux2, s.aux3, s.aux4, s.aux5})
        if (a) cudaStreamDestroy(a);
    if (s.stream) cudaStreamDestroy(s.stream);
    s = Slot();
}

// Binades (bit b: running value in [2^b, 2^(b+1)), ulp u = 2^(b-52)) in which adding one of the constants is an exact
// round-half-even tie: the constant's bits below u are exactly u/2, i.e. c * 2^(53-b) is an odd integer.  There the
// shift argument of the long-sequence path does not hold (the rounding depends on the parity of the sum), so its
// chunks in those binades are redone sequentially (long_kernel.cuh).
unsigned long long tie_binades(const double* c, int n)
{
    unsigned long long m = 0;
    for (int b = 0; b < 63; b++)
        for (int i = 0; i < n; i++) {
            if (!std::isfinite(c[i]) || c[i] == 0.0) continue;
            const double y = std::ldexp(std::fabs(c[i]), 53 - b);
            if (y < 9007199254740992.0 && y == std::floor(y) && std::fmod(y, 2.0) == 1.0) m |= 1ull << b;
        }
    return m;
}

// Fixed threshold of the long-sequence path for this ctx (0 = none): it needs every window to be far shorter than a
// protein.
int64_t effective_long_min(const plaac_ctx* ctx)
{
    if (ctx->long_min <= 0 || ctx->v2_nwr <= 0 || ctx->variant == 1) return 0;  // the path belongs to the v2 kernel
    const int64_t maxoff = std::max<int64_t>(std::max(4 * ctx->ks.w + 2, ctx->ks.core_len), ctx->ks.mw_window);
    return std::max<int64_t>(std::max<int64_t>(ctx->long_min, 1024), 4 * maxoff);
}

// Per-residue mode has a long-sequence path only beside the throughput kernels of residue_kernel_v2.cuh, and not when the
// window tracks come from generic_windows.cuh's protein-major kernels anyway (they need no help with long proteins, but
// the bookkeeping below assumes k_res_tracks).
bool long_res_ok(const plaac_ctx* ctx)
{
    return ctx->res_plan.ok && ctx->v2_nwr > 0 && ctx->variant != 1;
}

// Automatic threshold (long_min == -1).  The long-sequence path is a LATENCY device: whole CTAs per protein are far less
// efficient per residue than the bucketed kernel, so a protein goes there only if its sequential walk (~170 ns per
// residue in a lane of the bucketed kernel) would be a visible part of the batch's time, and only as many proteins
// as fit one wave of CTAs.  bins: k_long_levels' layout (or the host walk's).  Returns the threshold (0 = none) and
// the exact count / scratch size / longest remaining protein for it.
struct LongChoice {
    int64_t thr = 0, nlong = 0, scratch = 0, nbig = 0;  // nbig: of those, proteins of >= kLpBigMin residues
    int64_t lmax_rest = 0, n_hist_rest = 0;  // among proteins >= 1024 that stay on the bucketed path
};
LongChoice choose_long_threshold(const plaac_ctx* ctx, const unsigned long long* bins, int64_t ntotal, bool two_ctas = false)
{
    LongChoice c;
    const int64_t maxoff = std::max<int64_t>(std::max(4 * ctx->ks.w + 2, ctx->ks.core_len), ctx->ks.mw_window);
    const int64_t lb = std::max<int64_t>(std::max<int64_t>(1024, 4 * maxoff), ntotal / 81600 + 220);
    int64_t cnt = 0, scr = 0;
    int best = -1;
    for (int b = kLongBins - 1; b >= 0; b--) {  // suffix sums: proteins with len >= long_edge(b)
        if (long_edge(b) < lb) break;
        // (per-residue mode: k_long_post takes a whole SM per protein (190 KB of shared memory) and the bucketed kernels need
        // SMs beside it -- with records k_long_score's two CTAs per protein run too; measured on a yeast-sized set: 46 long
        // proteins 0.75 ms, 146: 0.78)
        if (cnt + (int64_t)bins[b] > (two_ctas ? ctx->sm_count / 2 : ctx->sm_count)) break;
        cnt += (int64_t)bins[b];
        if (long_edge(b) >= kLpBigMin) c.nbig += (int64_t)bins[b];
        scr += (int64_t)bins[kLongBins + b];
        best = b;
    }
    if (best >= 0 && cnt > 0 && ctx->v2_nwr > 0) {
        c.thr = long_edge(best);
        c.nlong = cnt;
        c.scratch = scr;
    } else
        c.nbig = 0;
    for (int b = 0; b < (c.thr ? best : kLongBins); b++) {
        if (!bins[b]) continue;
        c.lmax_rest = std::max<int64_t>(c.lmax_rest, (int64_t)bins[2 * kLongBins + b]);
        if (long_edge(b) >= kHistBins) c.n_hist_rest += (int64_t)bins[b];
    }
    return c;
}

// Enqueue the whole device pipeline for one batch on slot s.  d_offsets are absolute; off_base is
// subtracted to index d_codes.  Contains ONE stream synchronisation (the padded stream size).
// Exclusive scan out[0..n] of n int32 values on stream st: one CTA for small inputs, tiled (3 launches) for large ones.
int launch_scan(plaac_ctx* ctx, Slot& s, const int32_t* in, int64_t* out, int64_t n, cudaStream_t st)
{
    if (n <= 4 * kScanTile) {
        k_scan_exclusive<int32_t><<<1, 1024, 0, st>>>(in, out, n);
        ctx->stats.kernel_launches += 1;
        return PLAAC_OK;
    }
    const int64_t ntiles = (n + kScanTile - 1) / kScanTile;
    int rc;
    if ((rc = ensure(ctx, s.scan_tmp, sizeof(int64_t) * (size_t)(2 * ntiles + 2)))) return rc;
    int64_t* tile_sum = (int64_t*)s.scan_tmp.p;
    int64_t* tile_base = tile_sum + ntiles;
    k_scan_tile_sums<int32_t><<<(unsigned)ntiles, 1024, 0, st>>>(in, n, tile_sum);
    k_scan_exclusive<int64_t><<<1, 1024, 0, st>>>(tile_sum, tile_base, ntiles);
    k_scan_tiles_apply<int32_t><<<(unsigned)ntiles, 1024, 0, st>>>(in, n, tile_base, ntiles, out);
    ctx->stats.kernel_launches += 3;
    return PLAAC_OK;
}

// The segment kernels of a chunk (segments.cuh) on the slot's stream: with counts, k_seg_count[_long] and their scan
// into a.first first; then the bounds of the first a.cap segments and their scores.
int launch_segments(plaac_ctx* ctx, Slot& s, const SegArgs& a, int64_t np, bool counts)
{
    cudaStream_t st = s.stream;
    const unsigned gp = (unsigned)((np + 255) / 256);
    if (counts) {
        k_seg_count<<<gp, 256, 0, st>>>(a);
        ctx->stats.kernel_launches += 1;
        if (a.nlong > 0) {
            k_seg_count_long<<<(unsigned)a.nlong, kSegLongThreads, 0, st>>>(a);
            ctx->stats.kernel_launches += 1;
        }
        int rc = launch_scan(ctx, s, a.count, (int64_t*)a.first, np, st);
        if (rc) return rc;
    }
    if (a.cap > 0) {
        k_seg_bounds<<<gp, 256, 0, st>>>(a);
        ctx->stats.kernel_launches += 1;
        if (a.nlong > 0) {
            k_seg_bounds_long<<<(unsigned)a.nlong, kSegLongThreads, 0, st>>>(a);
            ctx->stats.kernel_launches += 1;
        }
        const unsigned gs = (unsigned)std::min<int64_t>((a.cap + 127) / 128, (int64_t)ctx->sm_count * 32);
        k_seg_score<<<gs, 128, 0, st>>>(a, np);
        ctx->stats.kernel_launches += 1;
    }
    CU(ctx, cudaGetLastError());
    return PLAAC_OK;
}

int run_batch(plaac_ctx* ctx, Slot& s, const uint8_t* d_codes, const int64_t* d_offsets, int64_t off_base,
              int64_t nprot, int64_t ntotal, plaac_summary* d_summaries, const plaac_residue_out* d_res,
              int64_t res_base, int64_t slots_bound = -1, int64_t nlong_known = -1, int64_t long_scratch_known = -1,
              int64_t long_thr_known = -1, int64_t nbig_known = -1, int64_t seg_cap = -1)
{
    if (nprot == 0) return PLAAC_OK;
    if (nprot > 0x7fffffff) return fail(ctx, PLAAC_E_INVALID, "more than 2^31-1 proteins in one device batch");
    cudaStream_t st = s.stream;
    const int64_t nbuckets = (nprot + 31) / 32;
    int rc;
    const bool use_v2 = ctx->variant >= 2 || (ctx->variant == 0 && ctx->v2_nwr > 0);  // v2 or v3: the role-split kernels
    // Long-sequence path: the throughput kernels only (summary mode: long_kernel.cuh; per-residue mode: long_residue.cuh
    // beside it, for the bucketed per-residue kernels of residue_kernel_v2.cuh).
    CU(ctx, cudaEventRecord(s.ev_a, st));
    const bool long_ok = use_v2 && (d_res ? long_res_ok(ctx) : d_summaries != nullptr);
    int64_t long_min = long_thr_known >= 0 ? long_thr_known : effective_long_min(ctx);
    if (long_ok && ctx->long_min < 0 && long_thr_known < 0 && ntotal >= 1024) {
        // automatic threshold with device-resident offsets: bin the lengths, let the host choose
        if ((rc = ensure(ctx, s.lg_bins, 3 * kLongBins * sizeof(unsigned long long)))) return rc;
        CU(ctx, cudaMemsetAsync(s.lg_bins.p, 0, 3 * kLongBins * sizeof(unsigned long long), st));
        k_long_levels<<<(unsigned)((nprot + 255) / 256), 256, 0, st>>>(d_offsets, nprot, (unsigned long long*)s.lg_bins.p);
        ctx->stats.kernel_launches += 1;
        CU(ctx, cudaMemcpyAsync(s.h_long, s.lg_bins.p, 3 * kLongBins * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        const LongChoice lc = choose_long_threshold(ctx, s.h_long, ntotal, d_res != nullptr);
        long_min = lc.thr;
        nlong_known = lc.nlong;
        long_scratch_known = lc.scratch;
        nbig_known = lc.nbig;
    }
    const bool use_long = long_ok && long_min > 0 && ntotal >= long_min && nlong_known != 0;
    const int64_t lm = use_long ? long_min : INT64_MAX;
    int64_t nlong = 0, long_scratch = 0, nbig = -1;
    if (use_long) {
        const int64_t cap = ntotal / long_min + 1;
        if ((rc = ensure(ctx, s.lg_list, sizeof(int32_t) * (size_t)cap))) return rc;
        if ((rc = ensure(ctx, s.lg_off, sizeof(int64_t) * (size_t)cap))) return rc;
        // [0] count, [1] scratch cursor, [2] count of >= kLpBigMin residues, [3] redone chunks (cumulative)
        if ((rc = ensure(ctx, s.lg_cnt, 32))) return rc;
        CU(ctx, cudaMemsetAsync(s.lg_cnt.p, 0, 24, st));
        k_long_select<<<(unsigned)((nprot + 255) / 256), 256, 0, st>>>(d_offsets, nprot, long_min, (int32_t*)s.lg_list.p,
                                                                      (int64_t*)s.lg_off.p, (unsigned long long*)s.lg_cnt.p,
                                                                      (int64_t)kLpBigMin);
        ctx->stats.kernel_launches += 1;
        if (nlong_known >= 0) {
            nlong = nlong_known;
            long_scratch = long_scratch_known;
            nbig = nbig_known;
        } else {
            CU(ctx, cudaMemcpyAsync(s.h_long, s.lg_cnt.p, 24, cudaMemcpyDeviceToHost, st));  // read after the sync below
        }
    }
    if ((rc = ensure(ctx, s.hist, sizeof(int32_t) * (kHistBins + 1)))) return rc;
    if ((rc = ensure(ctx, s.cursor, sizeof(int64_t) * (kHistBins + 2)))) return rc;
    if ((rc = ensure(ctx, s.order, sizeof(int32_t) * nprot))) return rc;
    if ((rc = ensure(ctx, s.nchunks, sizeof(int32_t) * nbuckets))) return rc;
    if ((rc = ensure(ctx, s.chunk_base, sizeof(int64_t) * (nbuckets + 1)))) return rc;

    CU(ctx, cudaMemsetAsync(s.hist.p, 0, sizeof(int32_t) * (kHistBins + 1), st));
    const int tb = 256;
    const unsigned g_hist = (unsigned)std::min<int64_t>(ctx->sm_count, (nprot + 4095) / 4096);
    const unsigned g_scat = (unsigned)std::min<int64_t>(ctx->sm_count, (nprot + kScatterTile - 1) / kScatterTile);
    k_len_hist<<<g_hist, kPrepThreads, kHistSmemBytes, st>>>(d_offsets, nprot, lm, (int32_t*)s.hist.p);
    k_scan_exclusive<int32_t><<<1, 1024, 0, st>>>((const int32_t*)s.hist.p, (int64_t*)s.cursor.p, kHistBins + 1);
    k_scatter<<<g_scat, kPrepThreads, kHistSmemBytes, st>>>(d_offsets, nprot, lm, (int64_t*)s.cursor.p, (int32_t*)s.order.p);
    const unsigned gb = (unsigned)((nbuckets * 32 + tb - 1) / tb);
    k_bucket_chunks<<<gb, tb, 0, st>>>(d_offsets, (const int32_t*)s.order.p, nprot, nbuckets, lm, (int32_t*)s.nchunks.p);
    if ((rc = launch_scan(ctx, s, (const int32_t*)s.nchunks.p, (int64_t*)s.chunk_base.p, nbuckets, st))) return rc;
    ctx->stats.kernel_launches += 4;
    CU(ctx, cudaMemcpyAsync(s.h_total, (int64_t*)s.chunk_base.p + nbuckets, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    int64_t slots = slots_bound;
    if (slots < 0) {
        // the caller knows nothing about the lengths (device-resident offsets): wait for the exact padded size
        CU(ctx, cudaStreamSynchronize(st));
        slots = *s.h_total;
        ctx->stats.last_padded_slots = slots * 32;
        if (use_long && nlong_known < 0) {
            nlong = (int64_t)s.h_long[0];
            long_scratch = (int64_t)s.h_long[1];
            nbig = (int64_t)s.h_long[2];
        }
    } else if (use_long && nlong_known < 0) {
        CU(ctx, cudaStreamSynchronize(st));
        nlong = (int64_t)s.h_long[0];
        long_scratch = (int64_t)s.h_long[1];
        nbig = (int64_t)s.h_long[2];
    }
    if ((rc = ensure(ctx, s.stream_buf, (size_t)std::max<int64_t>(slots, 1) * 32 * sizeof(uint4)))) return rc;
    if ((rc = ensure(ctx, s.tbw, (size_t)std::max<int64_t>(slots, 1) * 32 * sizeof(uint32_t)))) return rc;
    if ((rc = ensure(ctx, s.slot_bucket, (size_t)std::max<int64_t>(slots, 1) * sizeof(int32_t)))) return rc;

    // one block per 8 buckets, no grid-stride: buckets come in descending length, so handing them out as blocks retire is
    // longest-first list scheduling.  A resident grid with a stride gave the warps that own the first (longest) buckets
    // twice the average work (measured at 4 M proteins, time outside the scoring kernel: 1.28 ms with 5 CTAs per SM,
    // 1.17 with 8, 1.03 with 32).
    const unsigned pack_blocks = (unsigned)std::min<int64_t>((nbuckets + 7) / 8, 0x7fffffff);
    {
        auto pack = k_pack<false, false>;
        if (pack_is_std(ctx->ks.charge_plus, ctx->ks.charge_minus)) pack = ctx->ks.adjust_prolines ? k_pack<true, true> : k_pack<true, false>;
        pack<<<pack_blocks, 256, 0, st>>>(d_codes, d_offsets, off_base, (const int32_t*)s.order.p,
                                          (const int64_t*)s.chunk_base.p, nprot, nbuckets, lm, ctx->ks.adjust_prolines,
                                          ctx->ks.charge_plus, ctx->ks.charge_minus, (uint4*)s.stream_buf.p,
                                          (int32_t*)s.slot_bucket.p, (int*)s.errflag.p);
    }
    ctx->stats.kernel_launches += 1;

    BatchView bv;
    bv.stream = (const uint4*)s.stream_buf.p;
    bv.tbw = (uint32_t*)s.tbw.p;
    bv.order = (const int32_t*)s.order.p;
    bv.offsets = d_offsets;
    bv.chunk_base = (const int64_t*)s.chunk_base.p;
    bv.slot_bucket = (const int32_t*)s.slot_bucket.p;
    bv.nslots = slots;
    bv.nprot = nprot;
    bv.nbuckets = nbuckets;
    bv.off_base = off_base;
    bv.long_min = lm;

    if (d_summaries && use_v2) {
        if ((rc = ensure(ctx, s.core_list, sizeof(int32_t) * 2 * nprot))) return rc;
        if ((rc = ensure(ctx, s.core_count, 32))) return rc;  // [0] CORE list length, [8], [16] work-queue counters of the two roles
        CU(ctx, cudaMemsetAsync(s.core_count.p, 0, 32, st));
    }
    CU(ctx, cudaEventRecord(s.ev_b, st));
    bool long_launched = false;
    // The long-sequence path on streams of its own, launched first: its CTAs take SMs while the persistent CTAs of the
    // bucketed kernel start on the others and pick up the rest of the queue as SMs free up.  k_long_post (one thread-block
    // cluster per long protein) computes the per-residue arrays, or for records the forward score and the Viterbi parse;
    // with records, k_long_score computes the other columns beside it (two CTAs per protein), k_long_final the
    // Viterbi-dependent columns right behind the cluster kernel, and k_long_fix the two HMM scores when both are done.
    cudaStream_t long_st = d_res ? s.aux4 : s.aux1;
    if (use_long && nlong > 0) {
        if ((rc = ensure(ctx, s.lg_ext, (size_t)long_scratch + 256))) return rc;
        if ((rc = ensure(ctx, s.lg_ext_win, (size_t)long_scratch + 256))) return rc;
        if ((rc = ensure(ctx, s.lg_tb, (size_t)long_scratch + 256))) return rc;
        if ((rc = ensure(ctx, s.lg_vit, (size_t)long_scratch / 8 + 256))) return rc;
        LongArgs la;
        la.codes = d_codes;
        la.offsets = d_offsets;
        la.off_base = off_base;
        la.list = (const int32_t*)s.lg_list.p;
        la.scratch_off = (const int64_t*)s.lg_off.p;
        la.ks = ctx->ks;
        la.tabs = ctx->d_tabs;
        la.out = d_summaries;
        la.ext = (uint8_t*)s.lg_ext.p;
        la.ext_win = (uint8_t*)s.lg_ext_win.p;
        la.vit = (uint32_t*)s.lg_vit.p;
        la.errflag = (int*)s.errflag.p;
        for (int i = 0; i < 3; i++) la.tie_mask[i] = ctx->long_tie[1 + i];
        CU(ctx, cudaEventRecord(s.ev_fork, st));
        CU(ctx, cudaStreamWaitEvent(long_st, s.ev_fork, 0));
        const bool run_score = d_summaries != nullptr;
        if (run_score) {
            if ((rc = ensure(ctx, s.lg_hmm, sizeof(double) * 2 * (size_t)nlong))) return rc;
            if ((rc = ensure(ctx, s.lg_sum0, sizeof(double) * (size_t)nlong))) return rc;
            if ((rc = ensure(ctx, s.lg_vb, (size_t)long_scratch + 256))) return rc;
            la.sum0_out = (double*)s.lg_sum0.p;
            k_long_score<<<dim3((unsigned)nlong, 2), kLongThreads, sizeof(LongShared), long_st>>>(la);
            ctx->stats.kernel_launches += 1;
        }
        long_launched = true;
        ctx->stats.long_proteins += nlong;
        // one cluster per long protein, two size classes: posteriors + MAP parse (+ Viterbi parse), or, for records,
        // the forward score and the Viterbi parse
        if (d_res) {
            if ((rc = ensure(ctx, s.lp_s0, sizeof(double) * ((size_t)long_scratch + 256)))) return rc;
            if ((rc = ensure(ctx, s.lp_s1, sizeof(double) * ((size_t)long_scratch + 256)))) return rc;
            if ((rc = ensure(ctx, s.lp_lpseq, sizeof(double) * (size_t)nlong))) return rc;
        }
        const int64_t bnd_plane = long_scratch / 32 + 64;
        if ((rc = ensure(ctx, s.lp_bnd, sizeof(double) * (size_t)kLpBndPlanes * (size_t)bnd_plane))) return rc;
        LongPostArgs pa;
        pa.codes = d_codes;
        pa.offsets = d_offsets;
        pa.off_base = off_base;
        pa.res_base = res_base;
        pa.list = la.list;
        pa.scratch_off = la.scratch_off;
        pa.ks = ctx->ks;
        pa.tabs = ctx->d_tabs;
        if (d_res)
            pa.out = *d_res;
        else
            memset(&pa.out, 0, sizeof(pa.out));
        pa.S0 = d_res ? (double*)s.lp_s0.p : nullptr;
        pa.S1 = d_res ? (double*)s.lp_s1.p : nullptr;
        pa.bnd = (double*)s.lp_bnd.p;
        pa.bnd_plane = bnd_plane;
        pa.lpseq = d_res ? (double*)s.lp_lpseq.p : nullptr;
        pa.warm = std::max(1, std::abs(ctx->long_warm));
        pa.big_min = ctx->lp_big_min;
        pa.redone = (unsigned long long*)((char*)s.lg_cnt.p + 24);
        pa.want_post = d_res ? 1 : 0;
        pa.want_vit = (run_score || d_res->vit) ? 1 : 0;
        pa.hmm_out = run_score ? (double*)s.lg_hmm.p : nullptr;
        pa.vbytes = (run_score && !(d_res && d_res->vit)) ? (uint8_t*)s.lg_vb.p : nullptr;
        pa.tb = (uint8_t*)s.lg_tb.p;
        pa.vit_tie_mask = ctx->long_tie[0];
        pa.errflag = la.errflag;
        CU(ctx, cudaStreamWaitEvent(s.aux5, s.ev_fork, 0));
        if (pa.big_min != kLpBigMin) nbig = -1;  // (testing: the class counts are those of the default boundary)
        for (int cls = 0; cls < 2; cls++) {
            const int64_t ncls = nbig < 0 ? nlong : (cls ? nbig : nlong - nbig);
            if (ncls == 0) continue;
            pa.cluster = cls ? kLpBigCluster : 1;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(nlong * pa.cluster));
            cfg.blockDim = dim3(kLpThreads);
            cfg.dynamicSmemBytes = sizeof(LpShared);
            cfg.stream = s.aux5;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = (unsigned)pa.cluster;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            CU(ctx, cudaLaunchKernelEx(&cfg, k_long_post, pa));
            ctx->stats.kernel_launches += 1;
        }
        if (run_score) {
            k_long_final<<<(unsigned)nlong, kLongFinalThreads, 0, s.aux5>>>(la, (const uint8_t*)s.lg_vb.p, (d_res && d_res->vit) ? d_res->vit : nullptr, res_base);
            CU(ctx, cudaEventRecord(s.ev_j5, s.aux5));
            CU(ctx, cudaStreamWaitEvent(long_st, s.ev_j5, 0));
            k_long_fix<<<(unsigned)((nlong + 127) / 128), 128, 0, long_st>>>(la, (const double*)s.lg_hmm.p, (int)nlong);
            ctx->stats.kernel_launches += 2;
        }
    }
    if (d_summaries && use_v2) {
        V2Args g;
        g.bv = bv;
        g.ks = ctx->ks;
        g.tabs = ctx->d_tabs;
        g.out = d_summaries;
        g.ring_words = ctx->ring_words;
        g.nwr = ctx->v2_nwr;
        g.core_list = (int32_t*)s.core_list.p;
        g.core_count = (int32_t*)s.core_count.p;
        g.always_in = ctx->v2_always_in;
        g.work_counter = (unsigned long long*)((char*)s.core_count.p + 8);
        const bool use_v3 = ctx->variant != 2;
        if (use_v3) {
            const int full = 2 * ctx->ks.w + 1;
            g.ks_wfull = (double)(full * full);
            g.ks_cc2w = ctx->ks.cc2 * g.ks_wfull;
            g.ks_cc2full = ctx->ks.cc2 * (double)full;
            g.fi_a = ctx->ifold.a;
            g.fi_b = ctx->ifold.b;
            g.fi_c = ctx->ifold.c;
            g.fi_cfull = ctx->ifold.c * full;
            g.fi_cw = ctx->ifold.c * full * full;
        }
        const int64_t nitems = 2 * nbuckets, wpc = 2 * g.nwr;
        const unsigned grid = (unsigned)std::min<int64_t>((nitems + wpc - 1) / wpc, ctx->sm_count);  // 1 CTA per SM
        if (use_v3)
            v3_kernel(ctx->v3_opt)<<<grid, g.nwr * 64, ctx->v2_smem_bytes, st>>>(g);
        else
            k_score_summary_v2<<<grid, g.nwr * 64, ctx->v2_smem_bytes, st>>>(g);
        // masked stretches can be jumped exactly when the masking constant is a negative integer (it is -1e6)
        const double bn = ctx->ks.big_neg;
        if (bn < 0 && bn == std::floor(bn) && bn >= -4194304.0)
            k_core_search_jump<<<ctx->sm_count * 8, 128, 0, st>>>(bv, ctx->ks, ctx->d_tabs, d_summaries, g.core_list, g.core_count);
        else
            k_core_search<<<ctx->sm_count * 4, 128, 0, st>>>(bv, ctx->ks, ctx->d_tabs, d_summaries, g.core_list, g.core_count);
        ctx->stats.kernel_launches += 2;
        ctx->stats.score_launches += 1;
        if (long_launched && !d_res) {
            CU(ctx, cudaEventRecord(s.ev_j1, s.aux1));
            CU(ctx, cudaStreamWaitEvent(st, s.ev_j1, 0));
        }
    } else if (d_summaries) {
        const unsigned grid = (unsigned)((nbuckets + ctx->nwarps - 1) / ctx->nwarps);
        k_score_summary<<<grid, ctx->nwarps * 32, ctx->smem_bytes, st>>>(bv, ctx->ks, ctx->d_tabs, d_summaries,
                                                                         ctx->ring_words);
        ctx->stats.kernel_launches += 1;
        ctx->stats.score_launches += 1;
    }
    CU(ctx, cudaEventRecord(s.ev_c, st));
    if (d_res) {
        const bool res_v2 = ctx->res_plan.ok && ctx->v2_nwr > 0 && ctx->variant != 1;
        if (res_v2) {
            const size_t nslots = (size_t)std::max<int64_t>(slots, 1);
            if ((rc = ensure(ctx, s.res_b0, nslots * 512 * sizeof(double)))) return rc;
            if ((rc = ensure(ctx, s.res_b1, nslots * 512 * sizeof(double)))) return rc;
            if ((rc = ensure(ctx, s.res_a0, nslots * 512 * sizeof(double)))) return rc;
            if ((rc = ensure(ctx, s.res_a1, nslots * 512 * sizeof(double)))) return rc;
            if ((rc = ensure(ctx, s.res_mapw, nslots * 32 * sizeof(uint32_t)))) return rc;
            if ((rc = ensure(ctx, s.res_lpseq, (size_t)nbuckets * 32 * sizeof(double)))) return rc;
            ResArgs ra;
            ra.bv = bv;
            ra.ks = ctx->ks;
            ra.tabs = ctx->d_tabs;
            ra.out = *d_res;
            ra.res_base = res_base;
            ra.B0 = (double*)s.res_b0.p;
            ra.B1 = (double*)s.res_b1.p;
            ra.A0 = (double*)s.res_a0.p;
            ra.A1 = (double*)s.res_a1.p;
            ra.mapw = (uint32_t*)s.res_mapw.p;
            ra.lpseq = (double*)s.res_lpseq.p;
            TrackArgs ta;
            ta.codes = d_codes;
            ta.offsets = d_offsets;
            ta.off_base = off_base;
            ta.res_base = res_base;
            ta.nprot = nprot;
            ta.ks = ctx->ks;
            ta.tabs = ctx->d_tabs;
            ta.out = *d_res;
            ta.nx = ctx->res_plan.nx;
            ta.per_x = ctx->res_plan.per_x;
            ta.per_s = ctx->res_plan.per_s;
            ta.long_min = lm;
            ta.long_list = nullptr;
            if (long_launched) {
                // the eight tracks of the long proteins: the grid's warps share a protein's tiles (they only read the
                // residue codes; on the stream of the other tracks launch, ahead of it)
                TrackArgs tl = ta;
                tl.long_list = (const int32_t*)s.lg_list.p;
                CU(ctx, cudaStreamWaitEvent(s.aux3, s.ev_fork, 0));
                for (int64_t off = 0; off < nlong; off += 65535) {  // (gridDim.y is limited to 65535)
                    tl.long_list = (const int32_t*)s.lg_list.p + off;
                    k_res_tracks<<<dim3(16, (unsigned)std::min<int64_t>(65535, nlong - off)), kTrackWarps * 32, ctx->res_plan.trk_smem, s.aux3>>>(tl);
                    ctx->stats.kernel_launches += 1;
                }
            }
            rc = launch_residue_v2(ctx->res_plan, ra, ta, ctx->sm_count, st, s.aux1, s.aux2, s.aux3, s.ev_fork, s.ev_j1, s.ev_j2,
                                   s.ev_j3, &ctx->stats.kernel_launches);
        } else
            rc = launch_residue(ctx->ks, ctx->d_tabs, bv, *d_res, res_base, ctx->sm_count, st, &ctx->stats.kernel_launches);
        if (rc != PLAAC_OK) return fail(ctx, rc, "per-residue kernels failed to launch");
        if (long_launched) {
            CU(ctx, cudaEventRecord(s.ev_j4, s.aux4));
            CU(ctx, cudaEventRecord(s.ev_j5, s.aux5));
            CU(ctx, cudaStreamWaitEvent(st, s.ev_j4, 0));
            CU(ctx, cudaStreamWaitEvent(st, s.ev_j5, 0));
        }
    }
    if (ctx->generic_windows) {
        // everything that depends on the windows, tap by tap in the jar's order (generic_windows.cuh): into the caller's
        // per-residue arrays if there are any, else into scratch; then the window columns of the records
        GenArgs ga;
        ga.codes = d_codes;
        ga.offsets = d_offsets;
        ga.code_base = off_base;
        ga.nprot = nprot;
        ga.ww1 = ctx->params.ww1;
        ga.ww2 = ctx->params.ww2;
        ga.ww3 = ctx->params.ww3;
        ga.adjust_prolines = ctx->params.adjust_prolines ? 1 : 0;
        ga.cc0 = ctx->params.fi_cc[0];
        ga.cc1 = ctx->params.fi_cc[1];
        ga.cc2 = ctx->params.fi_cc[2];
        for (int c = 0; c < PLAAC_NAA; c++) {
            ga.t.hyd[c] = ctx->params.hydro2[c];
            ga.t.chg[c] = ctx->params.charge[c];
            ga.t.llr[c] = ctx->params.llr[c];
            ga.t.pap[c] = ctx->params.papa_lod[c];
        }
        const bool own = d_res && d_res->charge && d_res->hydro && d_res->fi && d_res->plaac && d_res->papa && d_res->fix2 &&
                         d_res->plaacx2 && d_res->papax2;
        if (own) {
            ga.out_base = res_base;
            ga.hydro = d_res->hydro, ga.charge = d_res->charge, ga.fi = d_res->fi, ga.plaac = d_res->plaac;
            ga.papa = d_res->papa, ga.fix2 = d_res->fix2, ga.plaacx2 = d_res->plaacx2, ga.papax2 = d_res->papax2;
        } else {
            const size_t N = (size_t)std::max<int64_t>(ntotal, 1);
            if ((rc = ensure(ctx, s.gen_f64, sizeof(double) * 8 * N))) return rc;
            double* d = (double*)s.gen_f64.p;
            ga.out_base = off_base;
            ga.hydro = d, ga.charge = d + N, ga.fi = d + 2 * N, ga.plaac = d + 3 * N;
            ga.papa = d + 4 * N, ga.fix2 = d + 5 * N, ga.plaacx2 = d + 6 * N, ga.papax2 = d + 7 * N;
        }
        ga.out = d_summaries;
        const unsigned gw = (unsigned)std::min<int64_t>((nprot + 3) / 4, (int64_t)ctx->sm_count * 64);
        k_gen_pass1<<<gw, 128, 0, st>>>(ga);
        k_gen_pass2<<<gw, 128, 0, st>>>(ga);
        ctx->stats.kernel_launches += 2;
        if (d_summaries) {
            k_gen_report<<<(unsigned)std::min<int64_t>((nprot + 127) / 128, (int64_t)ctx->sm_count * 16), 128, 0, st>>>(ga);
            ctx->stats.kernel_launches += 1;
        }
        if (d_res && !own) {
            // a caller that asked for some of the tracks only: hand those over from the scratch copy
            double* const dst[8] = {d_res->hydro, d_res->charge, d_res->fi, d_res->plaac, d_res->papa, d_res->fix2,
                                    d_res->plaacx2, d_res->papax2};
            const double* const src[8] = {ga.hydro, ga.charge, ga.fi, ga.plaac, ga.papa, ga.fix2, ga.plaacx2, ga.papax2};
            for (int k = 0; k < 8; k++)
                if (dst[k] && ntotal > 0)
                    CU(ctx, cudaMemcpyAsync(dst[k] + (off_base - res_base), src[k], sizeof(double) * (size_t)ntotal,
                                            cudaMemcpyDeviceToDevice, st));
        }
    }
    if (seg_cap >= 0 && d_summaries) {
        // segments (plaac_score_segments): both parses are final here -- the CORE search ran on st, and st has joined
        // the long-path streams
        if ((rc = ensure(ctx, s.sg_cnt, sizeof(int32_t) * (size_t)nprot))) return rc;
        if ((rc = ensure(ctx, s.sg_first, sizeof(int64_t) * (size_t)(nprot + 1)))) return rc;
        if ((rc = ensure(ctx, s.sg_ent, (3 * sizeof(int32_t) + sizeof(double)) * (size_t)std::max<int64_t>(seg_cap, 1)))) return rc;
        SegArgs a;
        a.bv = bv;
        a.codes = d_codes;
        a.tabs = ctx->d_tabs;
        a.long_list = long_launched ? (const int32_t*)s.lg_list.p : nullptr;
        a.long_off = long_launched ? (const int64_t*)s.lg_off.p : nullptr;
        a.long_vit = long_launched ? (const uint32_t*)s.lg_vit.p : nullptr;
        a.nlong = long_launched ? nlong : 0;
        a.count = (int32_t*)s.sg_cnt.p;
        a.first = (const int64_t*)s.sg_first.p;
        a.cap = seg_cap;
        double* ent = (double*)s.sg_ent.p;
        a.score = ent;
        a.prot = (int32_t*)(ent + seg_cap);
        a.start = a.prot + seg_cap;
        a.end = a.start + seg_cap;
        s.seg_args = a;
        s.seg_np = nprot;
        s.seg_cap = seg_cap;
        if ((rc = launch_segments(ctx, s, a, nprot, true))) return rc;
    }
    CU(ctx, cudaEventRecord(s.ev_d, st));
    CU(ctx, cudaGetLastError());
    s.timing_valid = true;
    return PLAAC_OK;
}

// Is this host pointer page-locked (cudaHostAlloc / cudaHostRegister) or otherwise known to the driver?
bool host_is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type != cudaMemoryTypeUnregistered;
}

int ensure_host(plaac_ctx* ctx, void*& p, size_t& cap, size_t bytes)
{
    if (bytes <= cap) return PLAAC_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 8 + 256;
    const cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        p = nullptr;
        return fail(ctx, PLAAC_E_NOMEM, "cudaHostAlloc(%zu bytes) for staging failed: %s", want, cudaGetErrorString(e));
    }
    cap = want;
    return PLAAC_OK;
}

// memcpy on several host threads: one thread moves 8-12 GB/s, a chunk's copy to or from a pageable caller buffer has to
// keep up with the 55 GB/s link
void par_memcpy(void* dst, const void* src, size_t n)
{
    constexpr size_t kMinPerThread = (size_t)8 << 20;
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t nt = std::min<size_t>(std::min<size_t>(hw ? hw : 1, 8), std::max<size_t>(1, n / kMinPerThread));
    if (nt <= 1) {
        memcpy(dst, src, n);
        return;
    }
    std::vector<std::thread> th;
    const size_t per = ((n + nt - 1) / nt + 4095) & ~(size_t)4095;
    for (size_t t = 1; t < nt; t++) {
        const size_t lo = std::min(n, t * per), hi = std::min(n, lo + per);
        if (hi <= lo) continue;
        try {
            th.emplace_back([=] { memcpy((char*)dst + lo, (const char*)src + lo, hi - lo); });
        } catch (...) {  // no thread to be had: this slice on the calling thread (nothing may throw across the C ABI)
            memcpy((char*)dst + lo, (const char*)src + lo, hi - lo);
        }
    }
    memcpy(dst, src, std::min(n, per));
    for (auto& t : th) t.join();
}

// Copies between PAGEABLE host memory and the device.  cudaMemcpy from pageable memory goes through the driver's own
// staging at a few GB/s; here chunks go through two pinned staging buffers of the ctx, filled / emptied by a
// multi-threaded memcpy while the other buffer's DMA runs (~20 GB/s).  Pinned caller memory is copied directly.
constexpr size_t kStageChunk = (size_t)32 << 20;

int stage_ready(plaac_ctx* ctx)
{
    for (int b = 0; b < 2; b++) {
        if (!ctx->stage_buf[b]) {
            const cudaError_t e = cudaHostAlloc(&ctx->stage_buf[b], kStageChunk, cudaHostAllocDefault);
            if (e != cudaSuccess) {
                cudaGetLastError();
                ctx->stage_buf[b] = nullptr;
                return fail(ctx, PLAAC_E_NOMEM, "cudaHostAlloc(staging): %s", cudaGetErrorString(e));
            }
        }
        if (!ctx->stage_ev[b]) CU(ctx, cudaEventCreateWithFlags(&ctx->stage_ev[b], cudaEventDisableTiming));
    }
    return PLAAC_OK;
}

// Returns when every byte of h_src has been read (the DMAs may still be in flight on st).
int h2d_any(plaac_ctx* ctx, void* d_dst, const void* h_src, size_t n, cudaStream_t st)
{
    if (n == 0) return PLAAC_OK;
    if (n < ((size_t)1 << 20) || host_is_pinned(h_src)) {
        CU(ctx, cudaMemcpyAsync(d_dst, h_src, n, cudaMemcpyHostToDevice, st));
        return PLAAC_OK;
    }
    int rc = stage_ready(ctx);
    if (rc) return rc;
    size_t off = 0;
    for (int i = 0; off < n; i++) {
        const int b = i & 1;
        const size_t len = std::min(kStageChunk, n - off);
        if (ctx->stage_pending[b]) CU(ctx, cudaEventSynchronize(ctx->stage_ev[b]));
        par_memcpy(ctx->stage_buf[b], (const char*)h_src + off, len);
        CU(ctx, cudaMemcpyAsync((char*)d_dst + off, ctx->stage_buf[b], len, cudaMemcpyHostToDevice, st));
        CU(ctx, cudaEventRecord(ctx->stage_ev[b], st));
        ctx->stage_pending[b] = true;
        off += len;
    }
    return PLAAC_OK;
}

// Returns when h_dst holds the data (pinned h_dst: when the copy is enqueued on st, as cudaMemcpyAsync).
int d2h_any(plaac_ctx* ctx, void* h_dst, const void* d_src, size_t n, cudaStream_t st)
{
    if (n == 0) return PLAAC_OK;
    if (n < ((size_t)1 << 20) || host_is_pinned(h_dst)) {
        CU(ctx, cudaMemcpyAsync(h_dst, d_src, n, cudaMemcpyDeviceToHost, st));
        return PLAAC_OK;
    }
    int rc = stage_ready(ctx);
    if (rc) return rc;
    const size_t nchunks = (n + kStageChunk - 1) / kStageChunk;
    auto enqueue = [&](size_t i) -> int {
        const int b = (int)(i & 1);
        const size_t off = i * kStageChunk, len = std::min(kStageChunk, n - off);
        if (ctx->stage_pending[b]) CU(ctx, cudaEventSynchronize(ctx->stage_ev[b]));
        CU(ctx, cudaMemcpyAsync(ctx->stage_buf[b], (const char*)d_src + off, len, cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaEventRecord(ctx->stage_ev[b], st));
        ctx->stage_pending[b] = true;
        return PLAAC_OK;
    };
    if ((rc = enqueue(0))) return rc;
    for (size_t i = 0; i < nchunks; i++) {
        if (i + 1 < nchunks && (rc = enqueue(i + 1))) return rc;  // (its buffer was emptied one iteration ago)
        const int b = (int)(i & 1);
        const size_t off = i * kStageChunk, len = std::min(kStageChunk, n - off);
        CU(ctx, cudaEventSynchronize(ctx->stage_ev[b]));
        ctx->stage_pending[b] = false;
        par_memcpy((char*)h_dst + off, ctx->stage_buf[b], len);
    }
    return PLAAC_OK;
}

int finish_slot(plaac_ctx* ctx, Slot& s)
{
    CU(ctx, cudaMemcpyAsync(s.h_err, s.errflag.p, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CU(ctx, cudaStreamSynchronize(s.stream));
    if (s.out_dst) {
        par_memcpy(s.out_dst, s.h_stage_sum, s.out_bytes);
        s.out_dst = nullptr;
    }
    ctx->stats.last_padded_slots = *s.h_total * 32;
    if (*s.h_err) {
        cudaMemsetAsync(s.errflag.p, 0, sizeof(int), s.stream);
        return fail(ctx, PLAAC_E_INVALID, "input contains residue codes > 21 or packed words >= 22^7 (treated as X)");
    }
    return PLAAC_OK;
}

}  // namespace

extern "C" {

int plaac_device_count(void)
try {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        g_last_error = std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e);
        cudaGetLastError();
        return 0;
    }
    return n;
} catch (...) {
    return api_caught(nullptr, "plaac_device_count");
}

int plaac_host_alloc(void** out, size_t bytes, int flags)
try {
    if (!out) return fail(nullptr, PLAAC_E_INVALID, "plaac_host_alloc: NULL argument");
    *out = nullptr;
    if (flags & ~PLAAC_HOST_WRITE_COMBINED) return fail(nullptr, PLAAC_E_INVALID, "plaac_host_alloc: unknown flags %d", flags);
    const unsigned f = cudaHostAllocPortable | ((flags & PLAAC_HOST_WRITE_COMBINED) ? cudaHostAllocWriteCombined : 0u);
    const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, f);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *out = nullptr;
        return fail(nullptr, e == cudaErrorMemoryAllocation ? PLAAC_E_NOMEM : PLAAC_E_CUDA, "cudaHostAlloc(%zu bytes): %s", bytes,
                    cudaGetErrorString(e));
    }
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_host_alloc");
}

int plaac_host_free(void* p)
try {
    if (!p) return PLAAC_OK;
    const cudaError_t e = cudaFreeHost(p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, PLAAC_E_INVALID, "cudaFreeHost: %s", cudaGetErrorString(e));
    }
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_host_free");
}

int plaac_host_register(void* p, size_t bytes)
try {
    if (!p || bytes == 0) return fail(nullptr, PLAAC_E_INVALID, "plaac_host_register: empty range");
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, e == cudaErrorMemoryAllocation ? PLAAC_E_NOMEM : PLAAC_E_INVALID, "cudaHostRegister(%zu bytes): %s",
                    bytes, cudaGetErrorString(e));
    }
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_host_register");
}

int plaac_host_unregister(void* p)
try {
    if (!p) return PLAAC_OK;
    const cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, PLAAC_E_INVALID, "cudaHostUnregister: %s", cudaGetErrorString(e));
    }
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_host_unregister");
}

int plaac_create(plaac_ctx** out, int device, const plaac_params* params)
try {
    if (!out || !params) return fail(nullptr, PLAAC_E_INVALID, "plaac_create: NULL argument");
    *out = nullptr;
    int ndev = plaac_device_count();
    if (ndev <= 0) return fail(nullptr, PLAAC_E_NODEVICE, "no CUDA device: %s", g_last_error.c_str());
    if (device < 0 || device >= ndev) return fail(nullptr, PLAAC_E_INVALID, "device %d out of range [0,%d)", device, ndev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, PLAAC_E_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return fail(nullptr, PLAAC_E_NODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    // (owned here until the very end: an exception on the way -- std::string, the table block -- must not leak the ctx)
    struct CtxGuard {
        plaac_ctx* p;
        ~CtxGuard() { if (p) plaac_destroy(p); }
    } guard{new plaac_ctx()};
    plaac_ctx* ctx = guard.p;
    ctx->device = device;
    ctx->params = *params;
    ctx->sm_count = prop.multiProcessorCount;
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    int rc = setup_scalars(ctx);
    if (rc != PLAAC_OK) {
        g_last_error = ctx->err;
        return rc;
    }
    auto bail = [&](int code) {
        g_last_error = ctx->err;
        return code;
    };
    if (cudaSetDevice(device) != cudaSuccess) {
        ctx->err = "cudaSetDevice failed";
        return bail(PLAAC_E_CUDA);
    }
    {
        std::unique_ptr<DeviceTables> h(new DeviceTables());
        fill_tables(ctx->params, *h, ctx->ks.w, (ctx->v3_opt & kV3IntFold) ? &ctx->ifold : nullptr);
        cudaError_t e = cudaMalloc((void**)&ctx->d_tabs, sizeof(DeviceTables));
        if (e == cudaSuccess) e = cudaMemcpy(ctx->d_tabs, h.get(), sizeof(DeviceTables), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            ctx->err = std::string("table upload: ") + cudaGetErrorString(e);
            return bail(PLAAC_E_CUDA);
        }
    }
    // (shared-memory limits are per function, not per ctx: common.cuh, raise_dynamic_smem_limit)
    {
        const int optin = (int)prop.sharedMemPerBlockOptin;
        const std::pair<const void*, size_t> fns[] = {{(const void*)k_long_score, sizeof(LongShared)},
                                                      {(const void*)k_long_post, sizeof(LpShared)},
                                                      {(const void*)k_score_summary, ctx->smem_bytes},
                                                      {(const void*)k_score_summary_v2, ctx->v2_smem_bytes},
                                                      {(const void*)k_len_hist, kHistSmemBytes},
                                                      {(const void*)k_scatter, kHistSmemBytes}};
        std::vector<std::pair<const void*, size_t>> all(std::begin(fns), std::end(fns));
        if (ctx->v2_nwr > 0) all.push_back({(const void*)v3_kernel(ctx->v3_opt), ctx->v2_smem_bytes});
        for (const auto& f : all) {
            const cudaError_t e = raise_dynamic_smem_limit(f.first, optin, f.second);
            if (e != cudaSuccess) {
                cudaGetLastError();
                ctx->err = std::string("shared-memory limit of a kernel: ") + cudaGetErrorString(e);
                return bail(PLAAC_E_CUDA);
            }
        }
    }
    {
        const plaac_params& P = ctx->params;
        double vc[4 + 2 * PLAAC_NAA];
        vc[0] = P.lt[0][0], vc[1] = P.lt[0][1], vc[2] = P.lt[1][0], vc[3] = P.lt[1][1];
        for (int i = 0; i < PLAAC_NAA; i++) vc[4 + i] = P.le[0][i], vc[4 + PLAAC_NAA + i] = P.le[1][i];
        ctx->long_tie[0] = tie_binades(vc, 4 + 2 * PLAAC_NAA);
        ctx->long_tie[1] = tie_binades(P.llr, PLAAC_NAA);
        ctx->long_tie[2] = tie_binades(P.le[0], PLAAC_NAA);
        ctx->long_tie[3] = tie_binades(P.hydro2, PLAAC_NAA);
    }
    // Two test hooks, and the library's only environment reads.  Each chooses which exact path of the long-sequence path
    // computes a value, so neither can change a result; they let tests reach paths that ordinary inputs reach only at
    // great cost.  PLAAC_LONG_TIES=1 marks every binade as a tie binade (every chunk is redone sequentially);
    // PLAAC_LP_BIG_MIN moves the boundary of k_long_post's cluster size class.
    if (const char* e = getenv("PLAAC_LONG_TIES"); e && strcmp(e, "1") == 0)
        for (unsigned long long& m : ctx->long_tie) m = ~0ull >> 1;
    if (const char* e = getenv("PLAAC_LP_BIG_MIN")) ctx->lp_big_min = atoll(e);
    ctx->res_plan = residue_v2_plan(ctx->ks);
    rc = residue_v2_setup(ctx->res_plan, (int)prop.sharedMemPerBlockOptin);
    if (rc == PLAAC_OK) rc = residue_setup(ctx->ks, ctx->ring_words);
    if (rc != PLAAC_OK) {
        ctx->err = "cudaFuncSetAttribute(per-residue kernels) failed";
        return bail(rc);
    }
    for (int i = 0; i < kSlots; i++) {
        rc = slot_init(ctx, ctx->slot[i]);
        if (rc != PLAAC_OK) return bail(rc);
    }
    guard.p = nullptr;
    *out = ctx;
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_create");
}

void plaac_destroy(plaac_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < kSlots; i++) slot_free(ctx->slot[i]);
    release(ctx->all_summaries);
    for (DevBuf* b : {&ctx->union_rec, &ctx->union_idx, &ctx->union_order, &ctx->union_out_idx, &ctx->var_ref, &ctx->var_ref_off, &ctx->var_wild, &ctx->null_counts,
                      &ctx->seq_scored, &ctx->seq_flags, &ctx->seq_live, &ctx->seq_pos, &ctx->seq_act[0], &ctx->seq_act[1]}) release(*b);
    for (int b = 0; b < 2; b++) {
        if (ctx->stage_buf[b]) cudaFreeHost(ctx->stage_buf[b]);
        if (ctx->stage_ev[b]) cudaEventDestroy(ctx->stage_ev[b]);
    }
    if (ctx->d_tabs) cudaFree(ctx->d_tabs);
    delete ctx;
}

const char* plaac_last_error(const plaac_ctx* ctx)
{
    return ctx ? ctx->err.c_str() : g_last_error.c_str();
}

int plaac_score_device(plaac_ctx* ctx, const uint8_t* d_codes, const int64_t* d_offsets, int64_t nprot, int64_t ntotal,
                       plaac_summary* d_summaries, const plaac_residue_out* d_per_res)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_device: NULL ctx");
    if (nprot < 0 || ntotal < 0) return fail(ctx, PLAAC_E_INVALID, "negative size");
    if (nprot == 0) return PLAAC_OK;
    if (!d_offsets || (!d_codes && ntotal > 0)) return fail(ctx, PLAAC_E_INVALID, "NULL codes/offsets");
    if (!d_summaries && !d_per_res) return fail(ctx, PLAAC_E_INVALID, "no output requested");
    CU(ctx, cudaSetDevice(ctx->device));
    ctx->last_slot = 0;
    return run_batch(ctx, ctx->slot[0], d_codes, d_offsets, 0, nprot, ntotal, d_summaries, d_per_res, 0);
} catch (...) {
    return api_caught(ctx, "plaac_score_device");
}

int plaac_sync(plaac_ctx* ctx)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_sync: NULL ctx");
    CU(ctx, cudaSetDevice(ctx->device));
    Slot& s = ctx->slot[0];
    int rc = finish_slot(ctx, s);
    if (s.timing_valid) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, s.ev_a, s.ev_d) == cudaSuccess) ctx->stats.last_total_ms = ms;
        if (cudaEventElapsedTime(&ms, s.ev_b, s.ev_c) == cudaSuccess) ctx->stats.last_score_ms = ms;
    }
    return rc;
} catch (...) {
    return api_caught(ctx, "plaac_sync");
}

void* plaac_stream(plaac_ctx* ctx)
{
    return ctx ? (void*)ctx->slot[0].stream : nullptr;
}

int plaac_set_chunk(plaac_ctx* ctx, int64_t max_residues, int64_t max_proteins)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_set_chunk: NULL ctx");
    if (max_residues < 0 || max_proteins < 0) return fail(ctx, PLAAC_E_INVALID, "negative chunk size");
    if (max_residues > 0) ctx->chunk_res = ctx->chunk_res_pr = max_residues;
    if (max_proteins > 0) ctx->chunk_prot = std::min<int64_t>(max_proteins, 0x7fffffff);
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_set_chunk");
}

int plaac_set_long_path(plaac_ctx* ctx, int64_t min_len, int warm)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_set_long_path: NULL ctx");
    if (min_len < -1) return fail(ctx, PLAAC_E_INVALID, "min_len must be -1 (automatic), 0 (off) or a length");
    ctx->long_min = min_len;
    if (warm != 0) ctx->long_warm = warm;
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_set_long_path");
}

int plaac_set_kernel_variant(plaac_ctx* ctx, int variant)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_set_kernel_variant: NULL ctx");
    if (variant < 0 || variant > 3) return fail(ctx, PLAAC_E_INVALID, "variant must be 0, 1, 2 or 3");
    if (variant >= 2 && ctx->v2_nwr <= 0)
        return fail(ctx, PLAAC_E_UNSUPPORTED, "v2/v3 kernel unavailable for these parameters: %s", ctx->v2_why.c_str());
    ctx->variant = variant;
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_set_kernel_variant");
}

int plaac_get_stats(plaac_ctx* ctx, plaac_stats* out)
try {
    if (!ctx || !out) return fail(ctx, PLAAC_E_INVALID, "plaac_get_stats: NULL argument");
    ctx->stats.long_redone_chunks = 0;
    for (int i = 0; i < kSlots; i++) {
        unsigned long long v = 0;
        if (ctx->slot[i].lg_cnt.p && cudaSetDevice(ctx->device) == cudaSuccess &&
            cudaMemcpy(&v, (char*)ctx->slot[i].lg_cnt.p + 24, sizeof(v), cudaMemcpyDeviceToHost) == cudaSuccess)
            ctx->stats.long_redone_chunks += (int64_t)v;
    }
    *out = ctx->stats;
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_get_stats");
}

void plaac_encode_host(const char* chars, int64_t n, uint8_t* codes)
{
    // aatoint, plaac.java:1508-1534: upper or lower case, '*' -> 21, everything else (incl. X) -> 0
    static const char names[] = "XACDEFGHIKLMNPQRSTVWY";
    uint8_t lut[256];
    memset(lut, 0, sizeof(lut));
    for (int i = 1; i <= 20; i++) {
        lut[(unsigned char)names[i]] = (uint8_t)i;
        lut[(unsigned char)(names[i] + 32)] = (uint8_t)i;
    }
    lut[(unsigned char)'*'] = 21;
    for (int64_t i = 0; i < n; i++) codes[i] = lut[(unsigned char)chars[i]];
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ ranking (N4)
namespace {

// One stable radix pass over the first n rows of buffer pair `cur`; the result lands in pair cur ^ 1.
template <bool SPLIT>
int rank_pass(plaac_ctx* ctx, Slot& s, int64_t n, int shift, int cur)
{
    const int64_t ntiles = (n + kRankTile - 1) / kRankTile;
    int rc;
    if ((rc = ensure(ctx, s.rk_hist, sizeof(int32_t) * (size_t)(kRankDigits * ntiles)))) return rc;
    if ((rc = ensure(ctx, s.rk_offs, sizeof(int64_t) * (size_t)(kRankDigits * ntiles + 1)))) return rc;
    cudaStream_t st = s.stream;
    k_rank_hist<SPLIT><<<(unsigned)ntiles, kRankThreads, 0, st>>>((const uint64_t*)s.rk_keys[cur].p, n, shift,
                                                                  (int32_t*)s.rk_hist.p, ntiles);
    if ((rc = launch_scan(ctx, s, (const int32_t*)s.rk_hist.p, (int64_t*)s.rk_offs.p, (int64_t)kRankDigits * ntiles, st))) return rc;
    k_rank_scatter<SPLIT><<<(unsigned)ntiles, kRankThreads, 0, st>>>(
        (const uint64_t*)s.rk_keys[cur].p, (const int32_t*)s.rk_vals[cur].p, (uint64_t*)s.rk_keys[cur ^ 1].p,
        (int32_t*)s.rk_vals[cur ^ 1].p, n, shift, (const int64_t*)s.rk_offs.p, ntiles);
    ctx->stats.kernel_launches += 2;
    CU(ctx, cudaGetLastError());
    return PLAAC_OK;
}

}  // namespace

extern "C" {

int plaac_rank_device(plaac_ctx* ctx, const plaac_summary* d_summaries, int64_t nprot, int flags, int32_t* d_order,
                      int64_t* n_core)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_rank_device: NULL ctx");
    if (nprot < 0 || nprot > 0x7fffffff) return fail(ctx, PLAAC_E_INVALID, "nprot out of range");
    if (flags != 0) return fail(ctx, PLAAC_E_INVALID, "flags are reserved and must be 0");
    if (n_core) *n_core = 0;
    if (nprot == 0) return PLAAC_OK;
    if (!d_summaries || !d_order) return fail(ctx, PLAAC_E_INVALID, "NULL summaries/order");
    CU(ctx, cudaSetDevice(ctx->device));
    Slot& s = ctx->slot[0];
    cudaStream_t st = s.stream;
    int rc;
    for (int k = 0; k < 2; k++) {
        if ((rc = ensure(ctx, s.rk_keys[k], sizeof(uint64_t) * (size_t)nprot))) return rc;
        if ((rc = ensure(ctx, s.rk_vals[k], sizeof(int32_t) * (size_t)nprot))) return rc;
    }
    const unsigned gk = (unsigned)((nprot + 255) / 256);
    int cur = 0;
    k_rank_keys<<<gk, 256, 0, st>>>(d_summaries, nprot, 0, (uint64_t*)s.rk_keys[cur].p,
                                    (int32_t*)s.rk_vals[cur].p);
    ctx->stats.kernel_launches += 1;
    for (int shift = 0; shift < 64; shift += 8) {
        if ((rc = rank_pass<false>(ctx, s, nprot, shift, cur))) return rc;
        cur ^= 1;
    }
    // CORE proteins first (stable), then order them by COREscore
    k_rank_keys<<<gk, 256, 0, st>>>(d_summaries, nprot, 1, (uint64_t*)s.rk_keys[cur].p, (int32_t*)s.rk_vals[cur].p);
    ctx->stats.kernel_launches += 1;
    if ((rc = rank_pass<true>(ctx, s, nprot, 0, cur))) return rc;
    cur ^= 1;
    const int64_t ntiles = (nprot + kRankTile - 1) / kRankTile;
    int64_t ncore = 0;  // rows with digit 0 = output base of (digit 1, tile 0)
    CU(ctx, cudaMemcpyAsync(&ncore, (const int64_t*)s.rk_offs.p + ntiles, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    if (ncore > 1) {
        // the tail (no CORE) must stay where it is: park it in d_order before the two buffers start to alternate
        const int tail_src = cur;
        if (nprot > ncore)
            CU(ctx, cudaMemcpyAsync(d_order + ncore, (const int32_t*)s.rk_vals[tail_src].p + ncore,
                                    sizeof(int32_t) * (size_t)(nprot - ncore), cudaMemcpyDeviceToDevice, st));
        for (int shift = 0; shift < 64; shift += 8) {
            if ((rc = rank_pass<false>(ctx, s, ncore, shift, cur))) return rc;
            cur ^= 1;
        }
        CU(ctx, cudaMemcpyAsync(d_order, s.rk_vals[cur].p, sizeof(int32_t) * (size_t)ncore, cudaMemcpyDeviceToDevice, st));
    } else {
        CU(ctx, cudaMemcpyAsync(d_order, s.rk_vals[cur].p, sizeof(int32_t) * (size_t)nprot, cudaMemcpyDeviceToDevice, st));
    }
    CU(ctx, cudaStreamSynchronize(st));
    if (n_core) *n_core = ncore;
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_rank_device");
}

int plaac_gather_device(plaac_ctx* ctx, const plaac_summary* d_summaries, const int32_t* d_order, int64_t count,
                        plaac_summary* d_out)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_gather_device: NULL ctx");
    if (count < 0) return fail(ctx, PLAAC_E_INVALID, "negative count");
    if (count == 0) return PLAAC_OK;
    if (!d_summaries || !d_order || !d_out) return fail(ctx, PLAAC_E_INVALID, "NULL argument");
    CU(ctx, cudaSetDevice(ctx->device));
    const int64_t threads = count * (int64_t)(sizeof(plaac_summary) / 8);
    k_rank_gather<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->slot[0].stream>>>(d_summaries, d_order, count, d_out);
    ctx->stats.kernel_launches += 1;
    CU(ctx, cudaGetLastError());
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_gather_device");
}

int plaac_rank(plaac_ctx* ctx, const plaac_summary* summaries, int64_t nprot, int flags, int32_t* order, int64_t* n_core)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_rank: NULL ctx");
    if (nprot < 0 || nprot > 0x7fffffff) return fail(ctx, PLAAC_E_INVALID, "nprot out of range");
    if (n_core) *n_core = 0;
    if (nprot == 0) return PLAAC_OK;
    if (!summaries || !order) return fail(ctx, PLAAC_E_INVALID, "NULL summaries/order");
    CU(ctx, cudaSetDevice(ctx->device));
    Slot& s = ctx->slot[0];
    int rc;
    if ((rc = ensure(ctx, s.summaries, sizeof(plaac_summary) * (size_t)nprot))) return rc;
    if ((rc = ensure(ctx, s.rk_order, sizeof(int32_t) * (size_t)nprot))) return rc;
    CU(ctx, cudaMemcpyAsync(s.summaries.p, summaries, sizeof(plaac_summary) * (size_t)nprot, cudaMemcpyHostToDevice, s.stream));
    if ((rc = plaac_rank_device(ctx, (const plaac_summary*)s.summaries.p, nprot, flags, (int32_t*)s.rk_order.p, n_core))) return rc;
    CU(ctx, cudaMemcpy(order, s.rk_order.p, sizeof(int32_t) * (size_t)nprot, cudaMemcpyDeviceToHost));
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_rank");
}

}  // extern "C"

namespace {

// Where k_shuffle_flags of a round of plaac_score_shuffles_seq (a slice of its list) writes: act = the slice of the
// device list (selection indices), flags = wpr words per (entry, column) row.
struct SeqRound {
    const int32_t* act;
    uint32_t* flags;
    int64_t wpr;
};

// What the host-buffer calls are given: one-byte codes + int64 offsets (plaac_score), radix-22 words + int32
// lengths (plaac_score_packed), a variant list over a reference batch of one-byte codes (plaac_score_variants), or
// shuffled replicates of that batch's proteins (plaac_score_shuffles).
struct HostInput {
    const uint8_t* codes = nullptr;
    const int64_t* offsets = nullptr;
    const uint32_t* words = nullptr;
    const int32_t* lengths = nullptr;
    int64_t nres = 0;  // packed input: the caller's total (checked against the lengths)
    int64_t pos0 = 0;  // packed input: residue index, counted from digit 0 of words[0], of the first protein (a shard of a
                       // larger batch starts in the middle of a word)
    const plaac_variants* var = nullptr;  // variant input: codes / offsets hold the nref proteins of the reference
    int64_t nref = 0;
    // shuffle input (over the reference, as var): replicate q = j * K + r is shuffle r of protein sel[j] (j for a NULL
    // sel), j < nsel; its output form is the per-protein tally of k_shuffle_tally into ctx->null_counts (and the rows of
    // nul->values), against the observed records in ctx->var_wild
    const plaac_null* nul = nullptr;  // nsel >= 0, proteins NULL for every protein; checked by plaac_score_shuffles
    // ... in a round of plaac_score_shuffles_seq: the replicates are r0 + [0, K) of each protein, the output form is the
    // round's hit flags (k_shuffle_flags), and the reference is already on the device
    int64_t r0 = 0;
    const SeqRound* seq = nullptr;
    bool packed() const { return words != nullptr || lengths != nullptr; }
};

// Variant or shuffle input: checks the reference, uploads it into the ctx buffers (once per call) and returns the total
// residue count of the variants or replicates.  Protein indices and first_sub are checked here, the substitutions
// during the chunk walk; a shuffle's selection is checked by plaac_score_shuffles.
int variants_prepare(plaac_ctx* ctx, const HostInput& in, int64_t& total)
{
    if (in.nref < 0) return fail(ctx, PLAAC_E_INVALID, "negative reference protein count");
    if (in.var) {
        const plaac_variants& V = *in.var;
        if (!V.protein || !V.first_sub || !V.pos || !V.code) return fail(ctx, PLAAC_E_INVALID, "NULL variant array with nvar = %lld", (long long)V.nvar);
    }
    if (!in.offsets) return fail(ctx, PLAAC_E_INVALID, "NULL reference offsets");
    for (int64_t i = 0; i < in.nref; i++)
        if (in.offsets[i + 1] < in.offsets[i]) return fail(ctx, PLAAC_E_INVALID, "reference offsets not monotone at protein %lld", (long long)i);
    const int64_t ref_base = in.offsets[0], ref_n = in.offsets[in.nref] - ref_base;
    if (ref_n > 0 && !in.codes) return fail(ctx, PLAAC_E_INVALID, "NULL reference codes");
    total = 0;
    if (in.nul) {
        const plaac_null& N = *in.nul;
        for (int64_t j = 0; j < N.nsel; j++) {
            const int64_t i = N.proteins ? N.proteins[j] : j;
            total += (in.offsets[i + 1] - in.offsets[i]) * N.replicates;
        }
    }
    const plaac_variants& V = in.var ? *in.var : plaac_variants{};
    if (in.var && V.first_sub[0] != 0) return fail(ctx, PLAAC_E_INVALID, "variant 0: first_sub[0] is %lld, not 0", (long long)V.first_sub[0]);
    for (int64_t v = 0; v < V.nvar; v++) {
        const int32_t p = V.protein[v];
        if (p < 0 || p >= in.nref)
            return fail(ctx, PLAAC_E_INVALID, "variant %lld: protein index %d outside [0, %lld)", (long long)v, p, (long long)in.nref);
        if (V.first_sub[v + 1] < V.first_sub[v])
            return fail(ctx, PLAAC_E_INVALID, "variant %lld: first_sub decreases (%lld after %lld)", (long long)v,
                        (long long)V.first_sub[v + 1], (long long)V.first_sub[v]);
        total += in.offsets[p + 1] - in.offsets[p];
    }
    if (in.seq) return PLAAC_OK;  // (a round of plaac_score_shuffles_seq: uploaded with its observed records)
    int rc;
    if ((rc = ensure(ctx, ctx->var_ref, (size_t)ref_n + 64))) return rc;
    if ((rc = ensure(ctx, ctx->var_ref_off, sizeof(int64_t) * (size_t)(in.nref + 1)))) return rc;
    // (every call blocks until done, so no earlier chunk still reads these buffers; the slots' streams start after this
    // synchronisation)
    cudaStream_t st = ctx->slot[0].stream;
    if ((rc = h2d_any(ctx, ctx->var_ref.p, in.codes + ref_base, (size_t)ref_n, st))) return rc;
    if ((rc = h2d_any(ctx, ctx->var_ref_off.p, in.offsets, sizeof(int64_t) * (size_t)(in.nref + 1), st))) return rc;
    CU(ctx, cudaStreamSynchronize(st));
    return PLAAC_OK;
}

// Substitutions [fs, fe) of variant v on a protein of len residues.
int check_subs(plaac_ctx* ctx, const plaac_variants& V, int64_t v, int64_t len)
{
    int64_t prev = -1;
    for (int64_t j = V.first_sub[v]; j < V.first_sub[v + 1]; j++) {
        const int64_t q = V.pos[j];
        if (q < 0 || q >= len)
            return fail(ctx, PLAAC_E_INVALID, "variant %lld: position %lld outside the protein (length %lld)", (long long)v,
                        (long long)q, (long long)len);
        if (q <= prev)
            return fail(ctx, PLAAC_E_INVALID, "variant %lld: positions do not strictly increase (%lld after %lld)",
                        (long long)v, (long long)q, (long long)prev);
        if (V.code[j] > 21)
            return fail(ctx, PLAAC_E_INVALID, "variant %lld: substitution code %d > 21", (long long)v, (int)V.code[j]);
        prev = q;
    }
    return PLAAC_OK;
}

// Compact ranked output of a whole host-buffer call: the records of every chunk were kept in ctx->all_summaries.
// on_device: the rows stay on the GPU (slot 0: `summaries` holds the hits->count ranked records, `rk_order` their indices
// in this call's batch) for plaac_score_multi_packed, which merges the shards' rows on one GPU.
int finish_hits(plaac_ctx* ctx, int64_t nprot, plaac_hits* hits, bool on_device = false)
{
    Slot& s = ctx->slot[0];
    cudaStream_t st = s.stream;
    const plaac_summary* all = (const plaac_summary*)ctx->all_summaries.p;
    int rc;
    hits->count = hits->n_core = 0;
    const int64_t cap = std::max<int64_t>(hits->capacity, 0);
    if ((rc = ensure(ctx, s.rk_order, sizeof(int32_t) * (size_t)nprot))) return rc;
    int32_t* d_order = (int32_t*)s.rk_order.p;
    int64_t count = 0;
    if (hits->mode == PLAAC_HITS_TOPK) {
        int64_t ncore = 0;
        if ((rc = plaac_rank_device(ctx, all, nprot, hits->rank_flags, d_order, &ncore))) return rc;
        hits->n_core = ncore;
        count = std::min(cap, nprot);
    } else {
        // rows with a CORE only: flag -> scan -> stable compaction, then the two stable LSD sorts of rank.cuh on those rows
        if ((rc = ensure(ctx, s.hit_flag, sizeof(int32_t) * (size_t)nprot))) return rc;
        if ((rc = ensure(ctx, s.hit_pos, sizeof(int64_t) * (size_t)(nprot + 1)))) return rc;
        const unsigned gn = (unsigned)((nprot + 255) / 256);
        k_hits_flag<<<gn, 256, 0, st>>>(all, nprot, (int32_t*)s.hit_flag.p);
        if ((rc = launch_scan(ctx, s, (const int32_t*)s.hit_flag.p, (int64_t*)s.hit_pos.p, nprot, st))) return rc;
        int64_t ncore = 0;
        CU(ctx, cudaMemcpyAsync(&ncore, (const int64_t*)s.hit_pos.p + nprot, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        ctx->stats.kernel_launches += 1;
        hits->n_core = ncore;
        count = std::min(cap, ncore);
        if (ncore > 0) {
            for (int k = 0; k < 2; k++) {
                if ((rc = ensure(ctx, s.rk_keys[k], sizeof(uint64_t) * (size_t)ncore))) return rc;
                if ((rc = ensure(ctx, s.rk_vals[k], sizeof(int32_t) * (size_t)ncore))) return rc;
            }
            int cur = 0;
            k_hits_compact<<<gn, 256, 0, st>>>((const int32_t*)s.hit_flag.p, (const int64_t*)s.hit_pos.p, nprot,
                                               (int32_t*)s.rk_vals[cur].p);
            ctx->stats.kernel_launches += 1;
            const unsigned gc = (unsigned)((ncore + 255) / 256);
            for (int field = 0; field < 2; field++) {
                k_hits_keys<<<gc, 256, 0, st>>>(all, (const int32_t*)s.rk_vals[cur].p, ncore, field, (uint64_t*)s.rk_keys[cur].p);
                ctx->stats.kernel_launches += 1;
                for (int shift = 0; shift < 64; shift += 8) {
                    if ((rc = rank_pass<false>(ctx, s, ncore, shift, cur))) return rc;
                    cur ^= 1;
                }
            }
            CU(ctx, cudaMemcpyAsync(d_order, s.rk_vals[cur].p, sizeof(int32_t) * (size_t)ncore, cudaMemcpyDeviceToDevice, st));
        }
    }
    hits->count = count;
    if (count > 0) {
        if (!on_device && !hits->records && !hits->index) return fail(ctx, PLAAC_E_INVALID, "plaac_hits: no output array");
        if (hits->records || on_device) {
            if ((rc = ensure(ctx, s.summaries, sizeof(plaac_summary) * (size_t)count))) return rc;
            if ((rc = plaac_gather_device(ctx, all, d_order, count, (plaac_summary*)s.summaries.p))) return rc;
            if (!on_device)
                CU(ctx, cudaMemcpyAsync(hits->records, s.summaries.p, sizeof(plaac_summary) * (size_t)count, cudaMemcpyDeviceToHost, st));
        }
        if (hits->index && !on_device)
            CU(ctx, cudaMemcpyAsync(hits->index, d_order, sizeof(int32_t) * (size_t)count, cudaMemcpyDeviceToHost, st));
    }
    CU(ctx, cudaStreamSynchronize(st));
    return PLAAC_OK;
}

// The effect output of a variant call (plaac_score_variant_effects): per variant, the selected columns of its record
// minus those of its wild type's.
struct EffectOut {
    uint32_t columns = 0;        // PLAAC_EFFECT_* mask, checked by the caller
    double* effects = nullptr;   // nvar x popcount(columns)
    plaac_summary* wild = nullptr;  // NULL or the reference's nref records
};

int score_host(plaac_ctx* ctx, const HostInput& in, int64_t nprot, plaac_summary* summaries, const plaac_residue_out* per_res,
               plaac_hits* hits, bool hits_on_device = false, const EffectOut* eff = nullptr, plaac_segments* seg = nullptr)
{
    if (nprot < 0) return fail(ctx, PLAAC_E_INVALID, "negative nprot");
    if (hits) {
        hits->count = hits->n_core = 0;
        if (hits->mode != PLAAC_HITS_CORE && hits->mode != PLAAC_HITS_TOPK) return fail(ctx, PLAAC_E_INVALID, "plaac_hits.mode must be PLAAC_HITS_CORE or PLAAC_HITS_TOPK");
        if (hits->capacity < 0) return fail(ctx, PLAAC_E_INVALID, "plaac_hits.capacity is negative");
        if (hits->rank_flags != 0) return fail(ctx, PLAAC_E_INVALID, "plaac_hits.rank_flags is reserved and must be 0");
        if (nprot > 0x7fffffff) return fail(ctx, PLAAC_E_INVALID, "more than 2^31-1 proteins with compact output");
    }
    if (nprot == 0) {
        if (in.packed() && in.nres != 0) return fail(ctx, PLAAC_E_INVALID, "nres does not equal the sum of the lengths");
        return PLAAC_OK;
    }
    const bool packed = in.packed();
    const plaac_variants* var = in.var;
    const plaac_null* nul = in.nul;
    if (var || nul) {
        if (per_res || hits) return fail(ctx, PLAAC_E_INVALID, "variants are scored in summary mode only");
    } else if (packed) {
        if (!in.lengths) return fail(ctx, PLAAC_E_INVALID, "NULL lengths");
        if (in.nres < 0 || (in.nres > 0 && !in.words)) return fail(ctx, PLAAC_E_INVALID, "NULL words / negative nres");
    } else {
        if (!in.offsets) return fail(ctx, PLAAC_E_INVALID, "NULL offsets");
        if (!in.codes && in.offsets[nprot] != in.offsets[0]) return fail(ctx, PLAAC_E_INVALID, "NULL codes");
    }
    if (!summaries && !per_res && !hits && !eff && !seg && !nul) return fail(ctx, PLAAC_E_INVALID, "no output requested");
    CU(ctx, cudaSetDevice(ctx->device));
    const bool want_rec = summaries || hits || eff || seg || nul;  // the device computes records
    int rc = PLAAC_OK;
    if (hits && (rc = ensure(ctx, ctx->all_summaries, sizeof(plaac_summary) * (size_t)nprot))) return rc;
    int64_t var_total = 0;
    if ((var || nul) && (rc = variants_prepare(ctx, in, var_total))) return rc;
    // Effects: the wild-type records are those of a plain call on the reference (so `wild` equals plaac_score's by
    // construction), uploaded into a device table that k_variant_effect reads.  Reference bytes > 21 make that call
    // return PLAAC_E_INVALID after writing its records; the variants are then scored all the same and the error is
    // returned at the end, as plaac_score returns it after the batch.
    const int ek = eff ? __builtin_popcount(eff->columns) : nul ? __builtin_popcount((uint32_t)nul->columns) : 0;
    const int64_t K = nul ? nul->replicates : 1;
    int rc_wild = PLAAC_OK;
    std::string err_wild;
    if (eff) {
        std::vector<plaac_summary> wild_host;
        plaac_summary* wild = eff->wild;
        if (!wild) {
            wild_host.resize((size_t)in.nref);
            wild = wild_host.data();
        }
        HostInput ref;
        ref.codes = in.codes;
        ref.offsets = in.offsets;
        rc_wild = score_host(ctx, ref, in.nref, wild, nullptr, nullptr);
        if (rc_wild != PLAAC_OK && rc_wild != PLAAC_E_INVALID) return rc_wild;
        err_wild = ctx->err;
        if ((rc = ensure(ctx, ctx->var_wild, sizeof(plaac_summary) * (size_t)in.nref))) return rc;
        cudaStream_t st = ctx->slot[0].stream;
        if ((rc = h2d_any(ctx, ctx->var_wild.p, wild, sizeof(plaac_summary) * (size_t)in.nref, st))) return rc;
        CU(ctx, cudaStreamSynchronize(st));
    }

    // Chunking: bounded device footprint; kSlots sets of buffers so the next chunks' H2D overlap this chunk's kernels and
    // D2H.  Chunk sizes ramp up from max/8 and down again towards the end: the first chunk's copy and the last chunk's
    // kernels + copy-back are the only parts of the pipeline nothing overlaps with.
    // (different half-widths of the windows: 64 bytes of track scratch per residue, so summary mode chunks like per-residue mode)
    const int64_t max_res_full = (per_res || ctx->generic_windows) ? std::min(ctx->chunk_res_pr, ctx->chunk_res) : ctx->chunk_res;
    const int64_t min_res = std::max<int64_t>(max_res_full / 8, 1 << 20);
    const int64_t first_off = packed || var || nul ? 0 : in.offsets[0];
    const int64_t total_res = var || nul ? var_total : packed ? in.nres : in.offsets[nprot] - first_off;
    int64_t ramp = min_res;
    const int64_t max_prot = ctx->chunk_prot;
    int64_t start = 0;
    const int64_t pos0 = packed ? in.pos0 : 0;
    int64_t pos = pos0;  // residue index of protein `start` (packed: counted from digit 0 of words[0])
    int which = 0;
    bool pending[kSlots] = {};
    // Pageable caller buffers (a Java heap array behind JNI, a std::vector): the driver would stage every copy
    // synchronously (measured 568 instead of 94 ms for the 4.4 G-residue shard).  The codes and the records then go
    // through pinned staging buffers of the slot, filled / emptied by a multi-threaded memcpy that overlaps the copies
    // and kernels of the other slots.
    const void* in_main = packed ? (const void*)in.words : (const void*)(in.codes + first_off);
    const bool stage_in = !var && !nul && total_res > 0 && !host_is_pinned(in_main);
    // (the host rows of the call: records, effects or null values)
    const void* out_rows = nul ? (const void*)nul->values : eff ? (const void*)eff->effects : (const void*)summaries;
    const size_t row_bytes = eff || nul ? sizeof(double) * (size_t)ek : sizeof(plaac_summary);
    const bool stage_sum = out_rows && !host_is_pinned(out_rows);
    // Segments: drained in chunk order, so seg_base is the number of segments of the proteins before the chunk.  A chunk
    // whose segments overflowed the slot's entries (and are wanted) reruns its bounds and score kernels with room for all
    // of them: the parse, codes and offsets are still in the slot.
    int64_t seg_base = 0;
    auto seg_drain = [&](Slot& s) -> int {
        const int64_t np = s.seg_np;
        s.seg_np = -1;
        const int64_t* hf = (const int64_t*)s.h_sg_first;
        const int64_t total = hf[np];
        for (int64_t i = 0; i < np; i++) seg->first[s.seg_p0 + i] = seg_base + hf[i];
        const int64_t want = std::min(total, std::max<int64_t>(seg->capacity - seg_base, 0));
        if (want > s.seg_cap) {
            int rc2;
            if ((rc2 = ensure(ctx, s.sg_ent, (3 * sizeof(int32_t) + sizeof(double)) * (size_t)total))) return rc2;
            SegArgs a = s.seg_args;
            double* ent = (double*)s.sg_ent.p;
            a.cap = total;
            a.score = ent;
            a.prot = (int32_t*)(ent + total);
            a.start = a.prot + total;
            a.end = a.start + total;
            if ((rc2 = launch_segments(ctx, s, a, np, false))) return rc2;
            if ((rc2 = ensure_host(ctx, s.h_sg_ent, s.h_sg_ent_cap, 16 * (size_t)total))) return rc2;
            CU(ctx, cudaMemcpyAsync(s.h_sg_ent, a.score, sizeof(double) * (size_t)total, cudaMemcpyDeviceToHost, s.stream));
            CU(ctx, cudaMemcpyAsync((double*)s.h_sg_ent + total, a.start, 2 * sizeof(int32_t) * (size_t)total, cudaMemcpyDeviceToHost, s.stream));
            CU(ctx, cudaStreamSynchronize(s.stream));
            s.seg_cap = total;
        }
        const double* hs = (const double*)s.h_sg_ent;
        const int32_t* hb = (const int32_t*)(hs + s.seg_cap);
        if (want > 0) {
            memcpy(seg->score + seg_base, hs, sizeof(double) * (size_t)want);
            memcpy(seg->start + seg_base, hb, sizeof(int32_t) * (size_t)want);
            memcpy(seg->end + seg_base, hb + s.seg_cap, sizeof(int32_t) * (size_t)want);
        }
        seg_base += total;
        return PLAAC_OK;
    };
    auto drain = [&](int i) -> int {
        if (!pending[i]) return PLAAC_OK;
        pending[i] = false;
        Slot& s = ctx->slot[i];
        int rcf = finish_slot(ctx, s);
        // (input bytes > 21: the chunk was scored in full, its segments are written like its records)
        if (seg && s.seg_np >= 0 && (rcf == PLAAC_OK || rcf == PLAAC_E_INVALID)) {
            const std::string keep = ctx->err;
            const int rcs = seg_drain(s);
            if (rcs != PLAAC_OK) return rcs;
            ctx->err = keep;
        }
        return rcf;
    };
    // Inside the chunk loop a CUDA error may not return at once: copies into the caller's buffers may be in flight on
    // other slots, and the header promises "blocks until done".  Errors break out to the drain loop below.
#define CUB(call)                                  \
    if ((rc = cu_rc(ctx, (call), #call)) != PLAAC_OK) break
    while (start < nprot && rc == PLAAC_OK) {
        // Cut the next chunk; validate it and collect what bounds its padded size while walking its lengths (the
        // walk overlaps the previous chunk's copies and kernels).
        int64_t end = start;
        const int64_t remaining = total_res - (pos - pos0);
        const int64_t max_res = std::min(max_res_full, std::max(min_res, std::min(ramp, remaining / 2)));
        ramp = std::min(max_res_full, ramp * 2);
        int64_t lmax = 0, nlong = 0, nlp = 0, lp_scratch = 0, nres = 0, nbigp = 0;
        const bool long_allowed = !per_res || long_res_ok(ctx);
        int64_t long_min = long_allowed ? effective_long_min(ctx) : 0;
        // (variants: always the automatic threshold -- at a fixed one, a saturation scan of a 10 000-residue protein would
        // send 190 000 equal-length variants to the latency path instead of the bucketed kernel)
        const bool long_auto = long_allowed && (ctx->long_min < 0 || var || nul) && ctx->v2_nwr > 0 && ctx->variant != 1;
        unsigned long long bins[3 * kLongBins];
        if (long_auto) memset(bins, 0, sizeof(bins));
        while (end < nprot && end - start < max_prot) {
            // (shuffles: a run of cnt replicates of one protein, so the walk is O(nsel + chunks), not O(nsel * K))
            int64_t cnt = 1;
            int64_t len;
            if (nul) {
                const int64_t j = end / K, i = nul->proteins ? nul->proteins[j] : j;
                len = in.offsets[i + 1] - in.offsets[i];
                cnt = std::min((j + 1) * K - end, max_prot - (end - start));
                if (len > 0) cnt = std::min(cnt, std::max<int64_t>((max_res - nres) / len, end == start));
                if (cnt == 0) break;
            } else {
                len = var ? in.offsets[var->protein[end] + 1] - in.offsets[var->protein[end]]
                          : packed ? (int64_t)in.lengths[end] : in.offsets[end + 1] - in.offsets[end];
            }
            if (len < 0) {
                rc = fail(ctx, PLAAC_E_INVALID, packed ? "negative length at protein %lld" : "offsets not monotone at protein %lld",
                          (long long)end);
                break;
            }
            if (len > 0x7fffff00LL) {
                rc = fail(ctx, PLAAC_E_INVALID, "protein %lld longer than 2^31", (long long)end);
                break;
            }
            if (end != start && nres + len > max_res) break;
            if (var && (rc = check_subs(ctx, *var, end, len))) break;
            if (long_auto && len >= 1024) {
                // decided after the walk (choose_long_threshold)
                const int b = long_bin(len);
                bins[b] += cnt;
                bins[kLongBins + b] += (unsigned long long)long_scratch_need(len) * cnt;
                bins[2 * kLongBins + b] = std::max<unsigned long long>(bins[2 * kLongBins + b], (unsigned long long)len);
            } else if (long_min > 0 && len >= long_min) {
                // scored by the long-sequence path; the bucketed stream sees an empty protein
                nlp += cnt;
                nbigp += (len >= kLpBigMin) * cnt;
                lp_scratch += long_scratch_need(len) * cnt;
            } else {
                lmax = std::max(lmax, len);
                nlong += (len >= kHistBins) * cnt;
            }
            nres += len * cnt;
            end += cnt;
        }
        if (rc != PLAAC_OK) break;
        if (packed && (pos - pos0) + nres > in.nres) {
            rc = fail(ctx, PLAAC_E_INVALID, "the lengths add up to more than nres = %lld residues", (long long)in.nres);
            break;
        }
        const int64_t np = end - start;
        int64_t long_thr = long_auto ? 0 : long_min;
        if (long_auto) {
            const LongChoice lc = choose_long_threshold(ctx, bins, nres, per_res != nullptr);
            long_thr = lc.thr;
            nlp = lc.nlong;
            nbigp = lc.nbig;
            lp_scratch = lc.scratch;
            lmax = std::max(lmax, lc.lmax_rest);
            nlong += lc.n_hist_rest;
        }
        // Upper bound of the bucketed stream (in 32-lane slots), so no host sync is needed for its size: proteins
        // are sorted by length, hence every bucket's longest member is no longer than the shortest member of the
        // bucket before it; only the first bucket and the buckets of unsorted >= 32768-residue proteins pay Lmax.
        const int64_t slots_bound = ((nlong + 31) / 32 + 2) * ((lmax + kChunk - 1) / kChunk) + (nres + 15 * np) / (32 * kChunk) + 1;
        Slot& s = ctx->slot[which];
        if ((rc = drain(which))) break;
        s.out_dst = nullptr;  // (a call that failed half-way may have left one behind)
        // packed input: words [w0, w1) hold the chunk; its first residue is digit `skip` of word w0
        const int64_t w0 = packed ? pos / PLAAC_PACK_PER_WORD : 0;
        const int64_t w1 = packed ? (pos + nres + PLAAC_PACK_PER_WORD - 1) / PLAAC_PACK_PER_WORD : 0;
        const int skip = packed ? (int)(pos - w0 * PLAAC_PACK_PER_WORD) : 0;
        const int64_t nwords = w1 - w0;
        {
            // k_pack reads whole aligned 16-byte blocks and masks what lies beyond a protein: keep the slack behind the
            // residues defined.  Zeroed once per (re)allocation, not per chunk: a memset between the two H2D copies of a
            // chunk sends the second one to the back of the copy engine's queue, behind the next chunk's codes
            // (measured: 94 -> 136 ms end to end for the 4.4 G-residue shard).
            const size_t cap0 = s.codes.cap;
            const size_t need = packed ? (size_t)((nwords + kUnpackTileWords) / kUnpackTileWords) * kUnpackTileBytes + 64 : (size_t)nres + 64;
            if ((rc = ensure(ctx, s.codes, need))) break;
            if (s.codes.cap != cap0) CUB(cudaMemsetAsync(s.codes.p, 0, s.codes.cap, s.stream));
        }
        if ((rc = ensure(ctx, s.offsets, sizeof(int64_t) * (np + 1)))) break;
        if (packed && (rc = ensure(ctx, s.words, sizeof(uint32_t) * (size_t)(nwords + 4)))) break;
        if ((packed || var || nul) && (rc = ensure(ctx, s.lengths, sizeof(int32_t) * (size_t)np))) break;
        // shuffles: the chunk's replicates are those of selected proteins [j0, j1]
        const int64_t j0 = nul ? start / K : 0, j1 = nul ? (end - 1) / K : -1;
        if (nul) {
            if ((rc = ensure(ctx, s.sh_rep, sizeof(ShuffleRep) * (size_t)np))) break;
            if (nul->proteins && (rc = ensure(ctx, s.v_prot, sizeof(int32_t) * (size_t)(j1 - j0 + 1)))) break;
        }
        const int64_t fs0 = var ? var->first_sub[start] : 0, nsub = var ? var->first_sub[end] - fs0 : 0;
        if (var) {
            if ((rc = ensure(ctx, s.v_prot, sizeof(int32_t) * (size_t)np))) break;
            if ((rc = ensure(ctx, s.v_first, sizeof(int64_t) * (size_t)(np + 1)))) break;
            if ((rc = ensure(ctx, s.v_pos, sizeof(int32_t) * (size_t)nsub))) break;
            if ((rc = ensure(ctx, s.v_code, (size_t)nsub))) break;
        }
        plaac_summary* d_sum = nullptr;
        if (hits)
            d_sum = (plaac_summary*)ctx->all_summaries.p + start;
        else if (summaries || eff || seg || nul) {
            if ((rc = ensure(ctx, s.summaries, sizeof(plaac_summary) * np))) break;
            d_sum = (plaac_summary*)s.summaries.p;
        }
        if ((eff || (nul && nul->values)) && (rc = ensure(ctx, s.v_effects, row_bytes * (size_t)np))) break;
        plaac_residue_out dres;
        if (per_res) {
            if ((rc = ensure(ctx, s.res_u8, (size_t)2 * (nres + 16)))) break;
            // (track arrays at multiples of 32 bytes: k_res_tracks3 then writes them with 256-bit stores)
            const size_t Np = ((size_t)nres + 3) & ~(size_t)3;
            if ((rc = ensure(ctx, s.res_f64, sizeof(double) * 10 * (Np + 4)))) break;
            uint8_t* u = (uint8_t*)s.res_u8.p;
            double* d = (double*)s.res_f64.p;
            const size_t N = (size_t)nres;
            dres.vit = u;
            dres.map = u + N;
            dres.charge = d;
            dres.hydro = d + Np;
            dres.fi = d + 2 * Np;
            dres.plaac = d + 3 * Np;
            dres.papa = d + 4 * Np;
            dres.fix2 = d + 5 * Np;
            dres.plaacx2 = d + 6 * Np;
            dres.papax2 = d + 7 * Np;
            dres.post_bg = d + 8 * Np;
            dres.post_prd = d + 9 * Np;
        }
        const void* src_main = packed ? (const void*)(in.words + w0) : (const void*)(in.codes + first_off + pos);
        const size_t main_bytes = packed ? sizeof(uint32_t) * (size_t)nwords : (size_t)nres;
        if (stage_in && main_bytes > 0) {
            if ((rc = ensure_host(ctx, s.h_stage_codes, s.h_stage_codes_cap, main_bytes))) break;
            par_memcpy(s.h_stage_codes, src_main, main_bytes);
            src_main = s.h_stage_codes;
        }
        if (stage_sum && (rc = ensure_host(ctx, s.h_stage_sum, s.h_stage_sum_cap, row_bytes * (size_t)np))) break;
        const uint8_t* d_codes = (const uint8_t*)s.codes.p;
        int64_t off_base = first_off + pos;  // offsets[] of the chunk are relative to this residue index
        if (var) {
            // only the chunk's slice of the variant list crosses the link; its residues are built from the reference
            CUB(cudaMemcpyAsync(s.v_prot.p, var->protein + start, sizeof(int32_t) * (size_t)np, cudaMemcpyHostToDevice, s.stream));
            CUB(cudaMemcpyAsync(s.v_first.p, var->first_sub + start, sizeof(int64_t) * (size_t)(np + 1), cudaMemcpyHostToDevice, s.stream));
            if (nsub > 0) {
                CUB(cudaMemcpyAsync(s.v_pos.p, var->pos + fs0, sizeof(int32_t) * (size_t)nsub, cudaMemcpyHostToDevice, s.stream));
                CUB(cudaMemcpyAsync(s.v_code.p, var->code + fs0, (size_t)nsub, cudaMemcpyHostToDevice, s.stream));
            }
            k_variant_lengths<<<(unsigned)((np + 255) / 256), 256, 0, s.stream>>>((const int32_t*)s.v_prot.p, np,
                                                                                  (const int64_t*)ctx->var_ref_off.p, (int32_t*)s.lengths.p);
            ctx->stats.kernel_launches += 1;
            if ((rc = launch_scan(ctx, s, (const int32_t*)s.lengths.p, (int64_t*)s.offsets.p, np, s.stream))) break;
            if (nres > 0) {
                k_variant_expand<<<(unsigned)((nres + kExpandTile - 1) / kExpandTile), kExpandThreads, 0, s.stream>>>(
                    (const uint8_t*)ctx->var_ref.p, (const int64_t*)ctx->var_ref_off.p, in.offsets[0], (const int32_t*)s.v_prot.p,
                    (const int64_t*)s.offsets.p, np, nres, (uint8_t*)s.codes.p);
                ctx->stats.kernel_launches += 1;
            }
            if (nsub > 0) {
                k_variant_apply<<<(unsigned)((nsub + 255) / 256), 256, 0, s.stream>>>((const int64_t*)s.v_first.p, fs0, np,
                                                                                     (const int32_t*)s.v_pos.p, (const uint8_t*)s.v_code.p,
                                                                                     nsub, (const int64_t*)s.offsets.p, (uint8_t*)s.codes.p);
                ctx->stats.kernel_launches += 1;
            }
            off_base = 0;
        } else if (nul) {
            const int32_t* d_sel = nullptr;
            if (nul->proteins) {
                CUB(cudaMemcpyAsync(s.v_prot.p, nul->proteins + j0, sizeof(int32_t) * (size_t)(j1 - j0 + 1), cudaMemcpyHostToDevice, s.stream));
                d_sel = (const int32_t*)s.v_prot.p;
            }
            k_shuffle_prep<<<(unsigned)((np + 255) / 256), 256, 0, s.stream>>>(d_sel, j0, start, K, in.r0, np, (const int64_t*)ctx->var_ref_off.p,
                                                                               nul->seed, (int32_t*)s.lengths.p, (ShuffleRep*)s.sh_rep.p);
            ctx->stats.kernel_launches += 1;
            if ((rc = launch_scan(ctx, s, (const int32_t*)s.lengths.p, (int64_t*)s.offsets.p, np, s.stream))) break;
            if (nres > 0) {
                k_shuffle_expand<<<(unsigned)((nres + kExpandTile - 1) / kExpandTile), kExpandThreads, 0, s.stream>>>(
                    (const uint8_t*)ctx->var_ref.p, (const ShuffleRep*)s.sh_rep.p, (const int64_t*)s.offsets.p, np, nres, (uint8_t*)s.codes.p);
                ctx->stats.kernel_launches += 1;
            }
            off_base = 0;
        } else if (packed) {
            if (main_bytes > 0) CUB(cudaMemcpyAsync(s.words.p, src_main, main_bytes, cudaMemcpyHostToDevice, s.stream));
            CUB(cudaMemcpyAsync(s.lengths.p, in.lengths + start, sizeof(int32_t) * (size_t)np, cudaMemcpyHostToDevice, s.stream));
            if (nwords > 0) {
                const int64_t ntiles = (nwords + kUnpackTileWords - 1) / kUnpackTileWords;
                const unsigned g = (unsigned)std::min<int64_t>((ntiles + 7) / 8, (int64_t)ctx->sm_count * 8);
                k_unpack22<<<g, kUnpackThreads, 0, s.stream>>>((const uint32_t*)s.words.p, nwords, (uint8_t*)s.codes.p, (int*)s.errflag.p);
                ctx->stats.kernel_launches += 1;
            }
            // offsets of the chunk = exclusive scan of its lengths, counted from the chunk's first residue
            if ((rc = launch_scan(ctx, s, (const int32_t*)s.lengths.p, (int64_t*)s.offsets.p, np, s.stream))) break;
            d_codes += skip;
            off_base = 0;
        } else {
            if (nres > 0) CUB(cudaMemcpyAsync(s.codes.p, src_main, (size_t)nres, cudaMemcpyHostToDevice, s.stream));
            CUB(cudaMemcpyAsync(s.offsets.p, in.offsets + start, sizeof(int64_t) * (np + 1), cudaMemcpyHostToDevice, s.stream));
        }
        // segment entries the slot keeps per chunk: several times the density of prion-like runs in proteomes (about
        // one per 10 000 residues); a denser chunk reruns its bounds and score kernels at drain
        const int64_t seg_cap = seg ? nres / 2048 + 1024 : -1;
        s.seg_np = -1;
        rc = run_batch(ctx, s, d_codes, (const int64_t*)s.offsets.p, off_base, np, nres, want_rec ? d_sum : nullptr,
                       per_res ? &dres : nullptr, off_base, slots_bound, nlp, lp_scratch, long_thr, nbigp, seg_cap);
        if (rc) break;
        if (seg) {
            s.seg_p0 = start;
            if ((rc = ensure_host(ctx, s.h_sg_first, s.h_sg_first_cap, sizeof(int64_t) * (size_t)(np + 1)))) break;
            if ((rc = ensure_host(ctx, s.h_sg_ent, s.h_sg_ent_cap, 16 * (size_t)seg_cap))) break;
            const SegArgs& a = s.seg_args;
            CUB(cudaMemcpyAsync(s.h_sg_first, a.first, sizeof(int64_t) * (size_t)(np + 1), cudaMemcpyDeviceToHost, s.stream));
            CUB(cudaMemcpyAsync(s.h_sg_ent, a.score, sizeof(double) * (size_t)seg_cap, cudaMemcpyDeviceToHost, s.stream));
            CUB(cudaMemcpyAsync((double*)s.h_sg_ent + seg_cap, a.start, 2 * sizeof(int32_t) * (size_t)seg_cap,
                                cudaMemcpyDeviceToHost, s.stream));
        }
        if (summaries && hits) {
            CUB(cudaMemcpyAsync(stage_sum ? (plaac_summary*)s.h_stage_sum : summaries + start, d_sum, sizeof(plaac_summary) * np,
                                cudaMemcpyDeviceToHost, s.stream));
        } else if (summaries) {
            CUB(cudaMemcpyAsync(stage_sum ? (plaac_summary*)s.h_stage_sum : summaries + start, s.summaries.p,
                                sizeof(plaac_summary) * np, cudaMemcpyDeviceToHost, s.stream));
        } else if (eff) {
            // the records stay on the device; only the chunk's np x ek effects cross the link
            k_variant_effect<<<(unsigned)((np * ek + 255) / 256), 256, 0, s.stream>>>(
                d_sum, (const plaac_summary*)ctx->var_wild.p, (const int32_t*)s.v_prot.p, np, eff->columns, (double*)s.v_effects.p);
            ctx->stats.kernel_launches += 1;
            CUB(cudaMemcpyAsync(stage_sum ? s.h_stage_sum : (void*)(eff->effects + start * ek), s.v_effects.p, row_bytes * (size_t)np,
                                cudaMemcpyDeviceToHost, s.stream));
        } else if (in.seq) {
            // (a round of plaac_score_shuffles_seq: the hits become flags, decided on by k_shuffle_stop after the round)
            k_shuffle_flags<<<(unsigned)((np * ek + 255) / 256), 256, 0, s.stream>>>(
                d_sum, (const plaac_summary*)ctx->var_wild.p, in.seq->act, start, K, np, (uint32_t)nul->columns, in.seq->wpr,
                in.seq->flags);
            ctx->stats.kernel_launches += 1;
        } else if (nul) {
            // the records stay on the device: the counts are summed there, and only the values rows (if any) cross the link
            double* d_val = nul->values ? (double*)s.v_effects.p : nullptr;
            k_shuffle_tally<<<(unsigned)((np * ek + 255) / 256), 256, 0, s.stream>>>(
                d_sum, (const plaac_summary*)ctx->var_wild.p, start, K, np, (uint32_t)nul->columns,
                (unsigned long long*)ctx->null_counts.p, d_val);
            ctx->stats.kernel_launches += 1;
            if (d_val)
                CUB(cudaMemcpyAsync(stage_sum ? s.h_stage_sum : (void*)(nul->values + start * ek), d_val, row_bytes * (size_t)np,
                                    cudaMemcpyDeviceToHost, s.stream));
        }
        if (out_rows && stage_sum) {
            s.out_dst = (char*)out_rows + row_bytes * (size_t)start;
            s.out_bytes = row_bytes * (size_t)np;
        }
        if (per_res && nres > 0) {
            const int64_t o = pos - pos0;
            const size_t N = (size_t)nres;
            uint8_t* hu[2] = {per_res->vit, per_res->map};
            const uint8_t* du[2] = {dres.vit, dres.map};
            for (int k = 0; k < 2; k++)
                if (hu[k] && rc == PLAAC_OK)
                    rc = cu_rc(ctx, cudaMemcpyAsync(hu[k] + o, du[k], N, cudaMemcpyDeviceToHost, s.stream), "cudaMemcpyAsync(per-residue bytes)");
            double* hd[10] = {per_res->charge, per_res->hydro,   per_res->fi,     per_res->plaac,   per_res->papa,
                              per_res->fix2,   per_res->plaacx2, per_res->papax2, per_res->post_bg, per_res->post_prd};
            const double* dd[10] = {dres.charge, dres.hydro,   dres.fi,     dres.plaac,   dres.papa,
                                    dres.fix2,   dres.plaacx2, dres.papax2, dres.post_bg, dres.post_prd};
            for (int k = 0; k < 10; k++)
                if (hd[k] && rc == PLAAC_OK)
                    rc = cu_rc(ctx, cudaMemcpyAsync(hd[k] + o, dd[k], N * sizeof(double), cudaMemcpyDeviceToHost, s.stream),
                               "cudaMemcpyAsync(per-residue doubles)");
        }
        pending[which] = true;  // (set even if a copy failed to enqueue: the drain below must still wait for this slot)
        if (rc) break;
        which = (which + 1) % kSlots;
        start = end;
        pos += nres;
    }
    for (int k = 0; k < kSlots; k++) {  // oldest chunk first
        const int rcd = drain((which + k) % kSlots);
        if (rc == PLAAC_OK) rc = rcd;
    }
#undef CUB
    if (rc == PLAAC_OK && packed && pos - pos0 != in.nres)
        rc = fail(ctx, PLAAC_E_INVALID, "the lengths add up to %lld residues, nres is %lld", (long long)(pos - pos0), (long long)in.nres);
    if (rc != PLAAC_OK) {
        // leave nothing behind that a later plaac_sync() could copy into this call's (by then stale) buffers
        const std::string keep = ctx->err;
        for (int k = 0; k < kSlots; k++) {
            cudaStreamSynchronize(ctx->slot[k].stream);
            ctx->slot[k].out_dst = nullptr;
        }
        cudaGetLastError();
        ctx->err = keep;
    }
    if (seg) {
        seg->first[start] = seg_base;  // (start == nprot unless the call failed part-way)
        seg->count = seg_base;
    }
    if (rc == PLAAC_OK && rc_wild != PLAAC_OK) {
        rc = rc_wild;
        ctx->err = err_wild;
    }
    if (hits && (rc == PLAAC_OK || (rc == PLAAC_E_INVALID && start >= nprot))) {
        // (invalid residue codes are reported after the batch, with every record computed: the compact output too)
        const std::string keep = ctx->err;
        const int rch = finish_hits(ctx, nprot, hits, hits_on_device);
        if (rch != PLAAC_OK)
            rc = rch;
        else
            ctx->err = keep;
    }
    return rc;
}

}  // namespace

extern "C" {

int plaac_score(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot, plaac_summary* summaries,
                const plaac_residue_out* per_res)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score: NULL ctx");
    HostInput in;
    in.codes = codes;
    in.offsets = offsets;
    if (nprot > 0 && !offsets) return fail(ctx, PLAAC_E_INVALID, "NULL offsets");
    if (nprot > 0 && !summaries && !per_res) return fail(ctx, PLAAC_E_INVALID, "no output requested");
    return score_host(ctx, in, nprot, summaries, per_res, nullptr);
} catch (...) {
    return api_caught(ctx, "plaac_score");
}

int plaac_score_hits(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot, plaac_hits* hits)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_hits: NULL ctx");
    if (!hits) return fail(ctx, PLAAC_E_INVALID, "plaac_score_hits: NULL hits");
    HostInput in;
    in.codes = codes;
    in.offsets = offsets;
    if (nprot > 0 && !offsets) return fail(ctx, PLAAC_E_INVALID, "NULL offsets");
    return score_host(ctx, in, nprot, nullptr, nullptr, hits);
} catch (...) {
    return api_caught(ctx, "plaac_score_hits");
}

int plaac_score_packed(plaac_ctx* ctx, const uint32_t* words, const int32_t* lengths, int64_t nprot, int64_t nres,
                       plaac_summary* summaries, const plaac_residue_out* per_res, plaac_hits* hits)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_packed: NULL ctx");
    HostInput in;
    in.words = words;
    in.lengths = lengths;
    in.nres = nres;
    if (nprot > 0 && !lengths) return fail(ctx, PLAAC_E_INVALID, "NULL lengths");
    return score_host(ctx, in, nprot, summaries, per_res, hits);
} catch (...) {
    return api_caught(ctx, "plaac_score_packed");
}

int plaac_score_variants(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                         const plaac_variants* variants, plaac_summary* summaries)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_variants: NULL ctx");
    if (!variants) return fail(ctx, PLAAC_E_INVALID, "plaac_score_variants: NULL variants");
    HostInput in;
    in.codes = codes;
    in.offsets = offsets;
    in.nref = nprot;
    in.var = variants;
    return score_host(ctx, in, variants->nvar, summaries, nullptr, nullptr);
} catch (...) {
    return api_caught(ctx, "plaac_score_variants");
}

int plaac_score_variant_effects(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                                const plaac_variants* variants, int32_t columns, double* effects, plaac_summary* wild)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_variant_effects: NULL ctx");
    if (!variants) return fail(ctx, PLAAC_E_INVALID, "plaac_score_variant_effects: NULL variants");
    if (columns <= 0 || columns >= (PLAAC_EFFECT_CORE_CHANGE << 1))
        return fail(ctx, PLAAC_E_INVALID, "plaac_score_variant_effects: columns 0x%x is not a non-empty set of PLAAC_EFFECT_* bits",
                    (unsigned)columns);
    if (variants->nvar > 0 && !effects) return fail(ctx, PLAAC_E_INVALID, "plaac_score_variant_effects: NULL effects with nvar = %lld",
                                                    (long long)variants->nvar);
    HostInput in;
    in.codes = codes;
    in.offsets = offsets;
    in.nref = nprot;
    in.var = variants;
    EffectOut eff;
    eff.columns = (uint32_t)columns;
    eff.effects = effects;
    eff.wild = wild;
    return score_host(ctx, in, variants->nvar, nullptr, nullptr, nullptr, false, &eff);
} catch (...) {
    return api_caught(ctx, "plaac_score_variant_effects");
}

int plaac_score_segments(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                         plaac_summary* summaries, plaac_segments* segments)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_segments: NULL ctx");
    if (!segments) return fail(ctx, PLAAC_E_INVALID, "plaac_score_segments: NULL segments");
    segments->count = 0;
    if (nprot < 0) return fail(ctx, PLAAC_E_INVALID, "negative nprot");
    if (segments->capacity < 0)
        return fail(ctx, PLAAC_E_INVALID, "plaac_score_segments: negative capacity %lld", (long long)segments->capacity);
    if (nprot > 0 && !segments->first) return fail(ctx, PLAAC_E_INVALID, "plaac_score_segments: NULL first with nprot = %lld", (long long)nprot);
    if (segments->capacity > 0 && (!segments->start || !segments->end || !segments->score))
        return fail(ctx, PLAAC_E_INVALID, "plaac_score_segments: NULL start, end or score with capacity = %lld",
                    (long long)segments->capacity);
    if (nprot > 0 && !offsets) return fail(ctx, PLAAC_E_INVALID, "NULL offsets");
    if (nprot == 0) {
        if (segments->first) segments->first[0] = 0;
        return PLAAC_OK;
    }
    HostInput in;
    in.codes = codes;
    in.offsets = offsets;
    return score_host(ctx, in, nprot, summaries, nullptr, nullptr, false, nullptr, segments);
} catch (...) {
    return api_caught(ctx, "plaac_score_segments");
}

int plaac_shuffle_host(const uint8_t* codes, int64_t n, uint64_t seed, int64_t protein, int64_t replicate, uint8_t* out)
try {
    if (n < 0 || n > 0x7fffffffLL) return fail(nullptr, PLAAC_E_INVALID, "plaac_shuffle_host: length %lld outside [0, 2^31)", (long long)n);
    if (protein < 0 || replicate < 0)
        return fail(nullptr, PLAAC_E_INVALID, "plaac_shuffle_host: negative protein %lld or replicate %lld", (long long)protein,
                    (long long)replicate);
    if (n > 0 && (!codes || !out)) return fail(nullptr, PLAAC_E_INVALID, "plaac_shuffle_host: NULL codes or out");
    const ShuffleKey k = shuffle_key(seed, protein, replicate, n);
    for (int64_t t = 0; t < n; t++) out[t] = codes[shuffle_index(k, (uint32_t)t)];
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_shuffle_host");
}

}  // extern "C"

namespace {

// The checks plaac_score_shuffles and plaac_score_shuffles_seq share (fn names the call in the messages).  nsel = the
// number of selected proteins (0: nothing to do), sel = the selection, NULL for every protein of the batch.
int null_check(plaac_ctx* ctx, const char* fn, int64_t nprot, const plaac_null& N, int64_t& nsel, const int32_t*& sel)
{
    const int64_t K = N.replicates;
    if (K < 0) return fail(ctx, PLAAC_E_INVALID, "%s: replicates %lld is negative", fn, (long long)K);
    if (N.nsel < -1) return fail(ctx, PLAAC_E_INVALID, "%s: nsel %lld is below -1", fn, (long long)N.nsel);
    if (N.reserved != 0) return fail(ctx, PLAAC_E_INVALID, "%s: reserved is %d, not 0", fn, (int)N.reserved);
    if (N.columns <= 0 || N.columns >= (PLAAC_NULL_HAS_CORE << 1))
        return fail(ctx, PLAAC_E_INVALID, "%s: columns 0x%x is not a non-empty set of bits 0..13", fn, (unsigned)N.columns);
    if (nprot < 0) return fail(ctx, PLAAC_E_INVALID, "negative nprot");
    if (N.nsel >= 0 && !N.proteins) return fail(ctx, PLAAC_E_INVALID, "%s: NULL proteins with nsel = %lld", fn, (long long)N.nsel);
    nsel = N.nsel < 0 ? nprot : N.nsel;
    if (nsel != 0 && !N.counts) return fail(ctx, PLAAC_E_INVALID, "%s: NULL counts with nsel = %lld", fn, (long long)N.nsel);
    sel = N.nsel < 0 ? nullptr : N.proteins;
    for (int64_t j = 0; sel && j < nsel; j++)
        if (sel[j] < 0 || sel[j] >= nprot)
            return fail(ctx, PLAAC_E_INVALID, "%s: selected protein %lld: index %d outside [0, %lld)", fn, (long long)j,
                        (int)sel[j], (long long)nprot);
    if (nsel == 0) return PLAAC_OK;
    if (nsel > 0x7fffffffLL) return fail(ctx, PLAAC_E_INVALID, "%s: more than 2^31-1 selected proteins", fn);
    if (K > INT64_MAX / nsel) return fail(ctx, PLAAC_E_INVALID, "%s: nsel x replicates overflows", fn);
    return PLAAC_OK;
}

// The checks of plaac_score_shuffles_seq and its multi-GPU form: null_check and the sequential call's own.
int seq_check(plaac_ctx* ctx, const char* fn, int64_t nprot, const plaac_null* null_spec, int64_t stop_hits,
              const int64_t* scored, int64_t& nsel, const int32_t*& sel)
{
    if (!null_spec) return fail(ctx, PLAAC_E_INVALID, "%s: NULL null_spec", fn);
    const plaac_null& N = *null_spec;
    if (stop_hits < 1) return fail(ctx, PLAAC_E_INVALID, "%s: stop_hits %lld is below 1", fn, (long long)stop_hits);
    if (N.values) return fail(ctx, PLAAC_E_INVALID, "%s: values must be NULL (the rows have unequal lengths)", fn);
    int rc = null_check(ctx, fn, nprot, N, nsel, sel);
    if (rc != PLAAC_OK) return rc;
    if (nsel != 0 && !scored) return fail(ctx, PLAAC_E_INVALID, "%s: NULL scored with nsel = %lld", fn, (long long)N.nsel);
    return PLAAC_OK;
}

// The observed records: the selection through the variant input form with no substitution, whose records equal
// plaac_score's.  Reference bytes > 21 make it return PLAAC_E_INVALID after writing them (rc_obs, err_obs); the
// replicates are then scored all the same and the error is returned at the end, as plaac_score returns it after the
// batch.  Then the tables the tallies read and sum into: the records in ctx->var_wild, nsel x k zero counts in
// ctx->null_counts.  Every slot's stream starts after this function's synchronisation.
int null_observed(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot, int64_t nsel, const int32_t* sel,
                  int k, plaac_summary* observed, int& rc_obs, std::string& err_obs)
{
    std::vector<int32_t> all;
    if (!sel) {
        all.resize((size_t)nsel);
        for (int64_t j = 0; j < nsel; j++) all[(size_t)j] = (int32_t)j;
    }
    std::vector<int64_t> no_sub((size_t)nsel + 1, 0);
    const int32_t no_pos = 0;
    const uint8_t no_code = 0;
    plaac_variants V = {nsel, sel ? sel : all.data(), no_sub.data(), &no_pos, &no_code};
    std::vector<plaac_summary> obs_host;
    plaac_summary* obs = observed;
    if (!obs) {
        obs_host.resize((size_t)nsel);
        obs = obs_host.data();
    }
    HostInput vin;
    vin.codes = codes;
    vin.offsets = offsets;
    vin.nref = nprot;
    vin.var = &V;
    rc_obs = score_host(ctx, vin, nsel, obs, nullptr, nullptr);
    if (rc_obs != PLAAC_OK && rc_obs != PLAAC_E_INVALID) return rc_obs;
    err_obs = ctx->err;

    const size_t count_bytes = sizeof(int64_t) * (size_t)nsel * (size_t)k;
    int rc;
    if ((rc = ensure(ctx, ctx->var_wild, sizeof(plaac_summary) * (size_t)nsel))) return rc;
    if ((rc = ensure(ctx, ctx->null_counts, count_bytes))) return rc;
    cudaStream_t st = ctx->slot[0].stream;
    if ((rc = h2d_any(ctx, ctx->var_wild.p, obs, sizeof(plaac_summary) * (size_t)nsel, st))) return rc;
    CU(ctx, cudaMemsetAsync(ctx->null_counts.p, 0, count_bytes, st));
    CU(ctx, cudaStreamSynchronize(st));
    return PLAAC_OK;
}

// The flag budget of a sequential null on ctx, in words: one bit per residue of a chunk's bound (plaac_set_chunk), so a
// test can make it small, and at least one word per column.
int64_t seq_budget(const plaac_ctx* ctx, int k) { return std::max<int64_t>(ctx->chunk_res / 32, k); }

// The span W = R_g - R_{g-1} of the round of a sequential null that starts at r0 = R_{g-1} (DESIGN.md sections 14 and
// 15).  W doubles (max(64, 4h) for the first round, or all of K when h > K / 4; r0 after it), but is at least wmin, so
// that a round holds at least one chunk bound of work on each GPU: a round's pipeline pays the latency of its first copy,
// its last chunk and its longest protein once, whatever its size.  A remainder K - R_g below wmin joins the round.  W is
// capped at the flag budget of one protein (wcap) and at K.
int64_t seq_span(int64_t K, int64_t r0, int64_t h, int64_t wmin, int64_t wcap)
{
    int64_t W = std::min(K - r0, std::max(r0 > 0 ? r0 : h > K / 4 ? K : std::max<int64_t>(64, 4 * h), wmin));
    if (K - r0 - W < wmin) W = K - r0;
    return std::min(W, wcap);
}

// ceil(chunk_res / res), res the residues of one replicate of every active protein
int64_t seq_wmin(int64_t chunk_res, int64_t res) { return (chunk_res + std::max<int64_t>(res, 1) - 1) / std::max<int64_t>(res, 1); }

// The rounds of plaac_score_shuffles_seq (DESIGN.md section 14), after null_observed.  At the end ctx->null_counts holds
// count and ctx->seq_scored L per (selection index, column).  Round g scores replicates [R_{g-1}, R_g) of the proteins
// still active, R_0 = 0, its span from seq_span with wmin = seq_wmin(chunk_res, res).  The hit flags take nact x k x W
// bits; where that exceeds the budget, the round runs as sub-rounds, each a slice of the same list over the round's whole
// span.  rc_rep, err_rep: PLAAC_E_INVALID and its message if a round reported reference bytes > 21 (it was scored in
// full).
int seq_rounds(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot, const plaac_null& N, int64_t nsel,
               const int32_t* sel, int k, int64_t h, int& rc_rep, std::string& err_rep)
{
    const int64_t K = N.replicates;
    Slot& s0 = ctx->slot[0];
    cudaStream_t st = s0.stream;
    const int64_t budget = seq_budget(ctx, k);
    const int64_t wcap = budget / k * 32;
    int rc;
    if ((rc = ensure(ctx, ctx->seq_scored, sizeof(int64_t) * (size_t)nsel * (size_t)k))) return rc;
    if ((rc = ensure(ctx, ctx->seq_live, sizeof(int32_t) * (size_t)nsel))) return rc;
    if ((rc = ensure(ctx, ctx->seq_pos, sizeof(int64_t) * (size_t)(nsel + 1)))) return rc;
    for (DevBuf& b : ctx->seq_act)
        if ((rc = ensure(ctx, b, sizeof(int32_t) * (size_t)(nsel + 1)))) return rc;
    // the round's list: its length, then selection indices (host act, device seq_act[cur]), and their reference indices
    std::vector<int32_t> act((size_t)nsel + 1), ref((size_t)nsel);
    act[0] = (int32_t)nsel;
    for (int64_t j = 0; j < nsel; j++) act[(size_t)j + 1] = (int32_t)j;
    if ((rc = h2d_any(ctx, ctx->seq_act[0].p, act.data(), sizeof(int32_t) * (size_t)(nsel + 1), st))) return rc;
    CU(ctx, cudaMemsetAsync(ctx->seq_scored.p, 0, sizeof(int64_t) * (size_t)nsel * (size_t)k, st));
    // the flags are zero between rounds (each sub-round clears what it set); a call that failed half-way may have left
    // some set
    if (ctx->seq_flags.cap > 0) CU(ctx, cudaMemsetAsync(ctx->seq_flags.p, 0, ctx->seq_flags.cap, st));
    CU(ctx, cudaStreamSynchronize(st));

    int cur = 0;
    int64_t nact = nsel, r0 = 0;
    while (nact > 0 && r0 < K) {
        int64_t res = 0;
        for (int64_t a = 0; a < nact; a++) {
            const int32_t j = act[(size_t)a + 1];
            ref[(size_t)a] = sel ? sel[j] : j;
            res += offsets[ref[(size_t)a] + 1] - offsets[ref[(size_t)a]];
        }
        const int64_t W = seq_span(K, r0, h, seq_wmin(ctx->chunk_res, res), wcap);
        const int64_t r1 = r0 + W, wpr = (W + 31) / 32;
        const int64_t per = std::max<int64_t>(1, budget / (k * wpr));  // entries per sub-round
        const int32_t* d_act = (const int32_t*)ctx->seq_act[cur].p + 1;
        int32_t* d_live = (int32_t*)ctx->seq_live.p;
        CU(ctx, cudaMemsetAsync(d_live, 0, sizeof(int32_t) * (size_t)nact, st));
        for (int64_t a0 = 0; a0 < nact; a0 += per) {
            const int64_t n = std::min(per, nact - a0);
            const size_t fbytes = sizeof(uint32_t) * (size_t)(n * k * wpr);
            const size_t cap0 = ctx->seq_flags.cap;
            if ((rc = ensure(ctx, ctx->seq_flags, fbytes))) return rc;
            if (ctx->seq_flags.cap != cap0) {
                CU(ctx, cudaMemsetAsync(ctx->seq_flags.p, 0, ctx->seq_flags.cap, st));
                CU(ctx, cudaStreamSynchronize(st));
            }
            const SeqRound sr = {d_act + a0, (uint32_t*)ctx->seq_flags.p, wpr};
            plaac_null R = N;
            R.replicates = W;
            R.nsel = n;
            R.proteins = ref.data() + a0;
            R.counts = nullptr;
            R.values = nullptr;
            HostInput in;
            in.codes = codes;
            in.offsets = offsets;
            in.nref = nprot;
            in.nul = &R;
            in.r0 = r0;
            in.seq = &sr;
            rc = score_host(ctx, in, n * W, nullptr, nullptr, nullptr);  // (returns with every slot synchronised)
            if (rc == PLAAC_E_INVALID && rc_rep == PLAAC_OK) {
                rc_rep = rc;
                err_rep = ctx->err;
            } else if (rc != PLAAC_OK && rc != PLAAC_E_INVALID) {
                return rc;
            }
            k_shuffle_stop<<<(unsigned)((n * k + 7) / 8), 256, 0, st>>>(sr.flags, sr.act, n, k, wpr, h, r0, r1, K,
                                                                       (int64_t*)ctx->null_counts.p, (int64_t*)ctx->seq_scored.p,
                                                                       d_live + a0);
            ctx->stats.kernel_launches += 1;
            CU(ctx, cudaMemsetAsync(sr.flags, 0, fbytes, st));
            // (the next sub-round's chunks run on the other slots' streams too)
            if (a0 + n < nact) CU(ctx, cudaStreamSynchronize(st));
        }
        // the next round's list, compacted on the device, comes back with one small copy
        int64_t* d_pos = (int64_t*)ctx->seq_pos.p;
        if ((rc = launch_scan(ctx, s0, d_live, d_pos, nact, st))) return rc;
        k_shuffle_compact<<<(unsigned)((nact + 255) / 256), 256, 0, st>>>(d_live, d_pos, d_act, nact, (int32_t*)ctx->seq_act[cur ^ 1].p);
        ctx->stats.kernel_launches += 1;
        CU(ctx, cudaMemcpyAsync(act.data(), ctx->seq_act[cur ^ 1].p, sizeof(int32_t) * (size_t)(nact + 1), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        nact = act[0];
        cur ^= 1;
        r0 = r1;
    }
    return PLAAC_OK;
}

}  // namespace

extern "C" {

int plaac_score_shuffles(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot, plaac_null* null_spec,
                         plaac_summary* observed)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_shuffles: NULL ctx");
    if (!null_spec) return fail(ctx, PLAAC_E_INVALID, "plaac_score_shuffles: NULL null_spec");
    const plaac_null& N = *null_spec;
    const int64_t K = N.replicates;
    int64_t nsel = 0;
    const int32_t* sel = nullptr;
    int rc = null_check(ctx, "plaac_score_shuffles", nprot, N, nsel, sel);
    if (rc != PLAAC_OK || nsel == 0) return rc;
    const int k = __builtin_popcount((uint32_t)N.columns);
    int rc_obs = PLAAC_OK;
    std::string err_obs;
    if ((rc = null_observed(ctx, codes, offsets, nprot, nsel, sel, k, observed, rc_obs, err_obs))) return rc;

    if (K > 0) {
        plaac_null R = N;
        R.nsel = nsel;
        R.proteins = sel;
        HostInput in;
        in.codes = codes;
        in.offsets = offsets;
        in.nref = nprot;
        in.nul = &R;
        rc = score_host(ctx, in, nsel * K, nullptr, nullptr, nullptr);
        if (rc != PLAAC_OK && rc != PLAAC_E_INVALID) return rc;
    }
    // (bytes > 21: the replicates were scored in full, so the counts are complete)
    const std::string keep = ctx->err;
    int rcc;
    cudaStream_t st = ctx->slot[0].stream;
    if ((rcc = d2h_any(ctx, N.counts, ctx->null_counts.p, sizeof(int64_t) * (size_t)nsel * (size_t)k, st))) return rcc;
    CU(ctx, cudaStreamSynchronize(st));
    ctx->err = keep;
    if (rc == PLAAC_OK && rc_obs != PLAAC_OK) {
        rc = rc_obs;
        ctx->err = err_obs;
    }
    return rc;
} catch (...) {
    return api_caught(ctx, "plaac_score_shuffles");
}

int plaac_score_shuffles_seq(plaac_ctx* ctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                             const plaac_null* null_spec, int64_t stop_hits, int64_t* scored, plaac_summary* observed)
try {
    const char* fn = "plaac_score_shuffles_seq";
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "%s: NULL ctx", fn);
    int64_t nsel = 0;
    const int32_t* sel = nullptr;
    int rc = seq_check(ctx, fn, nprot, null_spec, stop_hits, scored, nsel, sel);
    if (rc != PLAAC_OK || nsel == 0) return rc;
    const plaac_null& N = *null_spec;
    const int k = __builtin_popcount((uint32_t)N.columns);
    int rc_obs = PLAAC_OK;
    std::string err_obs;
    if ((rc = null_observed(ctx, codes, offsets, nprot, nsel, sel, k, observed, rc_obs, err_obs))) return rc;
    int rc_rep = PLAAC_OK;
    std::string err_rep;
    if ((rc = seq_rounds(ctx, codes, offsets, nprot, N, nsel, sel, k, stop_hits, rc_rep, err_rep))) return rc;
    const size_t bytes = sizeof(int64_t) * (size_t)nsel * (size_t)k;
    cudaStream_t st = ctx->slot[0].stream;
    if ((rc = d2h_any(ctx, N.counts, ctx->null_counts.p, bytes, st))) return rc;
    if ((rc = d2h_any(ctx, scored, ctx->seq_scored.p, bytes, st))) return rc;
    CU(ctx, cudaStreamSynchronize(st));
    // (bytes > 21: the replicates were scored in full, so counts and scored are complete)
    if (rc_rep != PLAAC_OK) {
        ctx->err = err_rep;
        return rc_rep;
    }
    if (rc_obs != PLAAC_OK) ctx->err = err_obs;
    return rc_obs;
} catch (...) {
    return api_caught(ctx, "plaac_score_shuffles_seq");
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ multi-GPU
#include <thread>

extern "C" {

int plaac_shard_plan(const int64_t* offsets, int64_t nprot, int nshards, int64_t* bounds)
try {
    if (!offsets || !bounds || nprot < 0 || nshards < 1) return PLAAC_E_INVALID;
    constexpr int64_t kPerProtein = 64;  // per-record overhead in residue equivalents
    const int64_t base = offsets[0];
    auto cost = [&](int64_t i) { return (offsets[i] - base) + kPerProtein * i; };  // monotone prefix cost
    const int64_t total = cost(nprot);
    bounds[0] = 0;
    for (int k = 1; k < nshards; k++) {
        const int64_t target = (int64_t)(((__int128)total * k) / nshards);
        int64_t lo = bounds[k - 1], hi = nprot;  // first i with cost(i) >= target
        while (lo < hi) {
            const int64_t mid = lo + (hi - lo) / 2;
            if (cost(mid) >= target)
                hi = mid;
            else
                lo = mid + 1;
        }
        bounds[k] = lo;
    }
    bounds[nshards] = nprot;
    return PLAAC_OK;
} catch (...) {
    return api_caught(nullptr, "plaac_shard_plan");
}

int plaac_score_multi(plaac_ctx* const* ctxs, int nctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                      plaac_summary* summaries, const plaac_residue_out* per_res)
try {
    if (!ctxs || nctx < 1) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_multi: no contexts");
    for (int k = 0; k < nctx; k++)
        if (!ctxs[k]) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_multi: NULL ctx %d", k);
    if (nctx == 1) return plaac_score(ctxs[0], codes, offsets, nprot, summaries, per_res);
    if (nprot < 0 || !offsets) return fail(ctxs[0], PLAAC_E_INVALID, "plaac_score_multi: bad offsets/nprot");
    if (nprot == 0) return PLAAC_OK;
    std::vector<int64_t> bounds((size_t)nctx + 1);
    plaac_shard_plan(offsets, nprot, nctx, bounds.data());
    std::vector<int> rcs((size_t)nctx, PLAAC_OK);
    std::vector<std::thread> threads;
    for (int k = 0; k < nctx; k++) {
        const int64_t lo = bounds[k], hi = bounds[k + 1];
        if (hi <= lo) continue;
        auto shard = [=, &rcs]() {
            plaac_residue_out shifted;
            const plaac_residue_out* pr = nullptr;
            if (per_res) {
                const int64_t o = offsets[lo] - offsets[0];
                shifted = *per_res;
                uint8_t** u8s[2] = {&shifted.vit, &shifted.map};
                for (auto p : u8s)
                    if (*p) *p += o;
                double** f64s[10] = {&shifted.charge, &shifted.hydro,   &shifted.fi,     &shifted.plaac,   &shifted.papa,
                                     &shifted.fix2,   &shifted.plaacx2, &shifted.papax2, &shifted.post_bg, &shifted.post_prd};
                for (auto p : f64s)
                    if (*p) *p += o;
                pr = &shifted;
            }
            rcs[k] = plaac_score(ctxs[k], codes, offsets + lo, hi - lo, summaries ? summaries + lo : nullptr, pr);
        };
        try {
            threads.emplace_back(shard);
        } catch (...) {  // no thread to be had: this shard on the calling thread (nothing may throw across the C ABI)
            shard();
        }
    }
    for (auto& t : threads) t.join();
    for (int k = 0; k < nctx; k++)
        if (rcs[k] != PLAAC_OK) return rcs[k];
    return PLAAC_OK;
} catch (...) {
    return api_caught((ctxs && nctx > 0 ? ctxs[0] : nullptr), "plaac_score_multi");
}

int plaac_score_multi_packed(plaac_ctx* const* ctxs, int nctx, const uint32_t* words, const int32_t* lengths, int64_t nprot,
                             int64_t nres, plaac_summary* summaries, const plaac_residue_out* per_res, plaac_hits* hits)
try {
    if (!ctxs || nctx < 1) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_multi_packed: no contexts");
    for (int k = 0; k < nctx; k++)
        if (!ctxs[k]) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_multi_packed: NULL ctx %d", k);
    if (nctx == 1) return plaac_score_packed(ctxs[0], words, lengths, nprot, nres, summaries, per_res, hits);
    plaac_ctx* c0 = ctxs[0];
    if (nprot < 0 || (nprot > 0 && !lengths)) return fail(c0, PLAAC_E_INVALID, "plaac_score_multi_packed: bad lengths/nprot");
    if (hits) {
        hits->count = hits->n_core = 0;
        if (hits->mode != PLAAC_HITS_CORE && hits->mode != PLAAC_HITS_TOPK) return fail(c0, PLAAC_E_INVALID, "plaac_hits.mode must be PLAAC_HITS_CORE or PLAAC_HITS_TOPK");
        if (hits->capacity < 0 || nprot > 0x7fffffff) return fail(c0, PLAAC_E_INVALID, "plaac_hits: bad capacity / too many proteins");
        if (hits->rank_flags != 0) return fail(c0, PLAAC_E_INVALID, "plaac_hits.rank_flags is reserved and must be 0");
    }
    if (nprot == 0) return nres == 0 ? PLAAC_OK : fail(c0, PLAAC_E_INVALID, "nres does not equal the sum of the lengths");
    // Shard bounds balanced on residues + 64 per protein (as plaac_shard_plan).  The prefix over the lengths is taken on
    // several host threads: block sums first, then every block finds the bounds that fall into it.
    std::vector<int64_t> bounds((size_t)nctx + 1, nprot), rpos((size_t)nctx + 1, nres);
    {
        constexpr int64_t kPerProtein = 64;
        const int nb = (int)std::max<int64_t>(1, std::min<int64_t>(16, nprot / (1 << 20)));
        const int64_t per = (nprot + nb - 1) / nb;
        std::vector<int64_t> bsum((size_t)nb, 0);
        std::vector<int> bneg((size_t)nb, 0);
        auto block = [&](int b) {
            const int64_t lo = std::min(nprot, b * per), hi = std::min(nprot, lo + per);
            int64_t t = 0;
            int neg = 0;
            for (int64_t i = lo; i < hi; i++) {
                neg |= lengths[i] < 0;
                t += lengths[i];
            }
            bsum[(size_t)b] = t;
            bneg[(size_t)b] = neg;
        };
        {
            std::vector<std::thread> th;
            for (int b = 1; b < nb; b++) th.emplace_back(block, b);
            block(0);
            for (auto& t : th) t.join();
        }
        int64_t tot = 0;
        for (int b = 0; b < nb; b++) {
            if (bneg[(size_t)b]) return fail(c0, PLAAC_E_INVALID, "negative length in the batch");
            tot += bsum[(size_t)b];
        }
        if (tot != nres) return fail(c0, PLAAC_E_INVALID, "the lengths add up to %lld residues, nres is %lld", (long long)tot, (long long)nres);
        const int64_t total = tot + kPerProtein * nprot;
        bounds[0] = 0;
        rpos[0] = 0;
        int k = 1;
        int64_t r = 0;  // residues before the current block
        for (int b = 0; b < nb && k < nctx; b++) {
            const int64_t lo = std::min(nprot, b * per), hi = std::min(nprot, lo + per);
            const int64_t cost_end = (r + bsum[(size_t)b]) + kPerProtein * hi;
            int64_t i = lo, rr = r;
            // first i with cost(i) >= target_k, for every target that is reached inside this block
            while (k < nctx && (int64_t)(((__int128)total * k) / nctx) <= cost_end) {
                const int64_t target = (int64_t)(((__int128)total * k) / nctx);
                while (i < hi && rr + kPerProtein * i < target) rr += lengths[i++];
                if (i >= hi && rr + kPerProtein * i < target) break;  // reached in a later block
                bounds[(size_t)k] = i;
                rpos[(size_t)k] = rr;
                k++;
            }
            r += bsum[(size_t)b];
        }
        bounds[(size_t)nctx] = nprot;
        rpos[(size_t)nctx] = nres;
    }
    std::vector<int> rcs((size_t)nctx, PLAAC_OK);
    std::vector<plaac_hits> sh_hits((size_t)nctx);
    std::vector<std::thread> threads;
    for (int k = 0; k < nctx; k++) {
        const int64_t lo = bounds[(size_t)k], hi = bounds[(size_t)k + 1];
        if (hi <= lo) continue;
        if (hits) {
            sh_hits[(size_t)k] = *hits;
            sh_hits[(size_t)k].capacity = std::min<int64_t>(hits->capacity, hi - lo);
            sh_hits[(size_t)k].records = nullptr;  // the shard's rows stay on its GPU (finish_hits, on_device)
            sh_hits[(size_t)k].index = nullptr;
        }
        auto shard = [=, &rcs, &sh_hits, &rpos]() {
            plaac_residue_out shifted;
            const plaac_residue_out* pr = nullptr;
            if (per_res) {
                const int64_t o = rpos[(size_t)k];
                shifted = *per_res;
                uint8_t** u8s[2] = {&shifted.vit, &shifted.map};
                for (auto p : u8s)
                    if (*p) *p += o;
                double** f64s[10] = {&shifted.charge, &shifted.hydro,   &shifted.fi,     &shifted.plaac,   &shifted.papa,
                                     &shifted.fix2,   &shifted.plaacx2, &shifted.papax2, &shifted.post_bg, &shifted.post_prd};
                for (auto p : f64s)
                    if (*p) *p += o;
                pr = &shifted;
            }
            HostInput in;
            const int64_t w0 = rpos[(size_t)k] / PLAAC_PACK_PER_WORD;
            in.words = words + w0;
            in.lengths = lengths + lo;
            in.nres = rpos[(size_t)k + 1] - rpos[(size_t)k];
            in.pos0 = rpos[(size_t)k] - w0 * PLAAC_PACK_PER_WORD;
            try {
                rcs[(size_t)k] = score_host(ctxs[k], in, hi - lo, summaries ? summaries + lo : nullptr, pr,
                                            hits ? &sh_hits[(size_t)k] : nullptr, /*hits_on_device=*/true);
            } catch (...) {
                rcs[(size_t)k] = api_caught(ctxs[k], "plaac_score_multi_packed (shard)");
            }
        };
        try {
            threads.emplace_back(shard);
        } catch (...) {  // no thread to be had: this shard on the calling thread (nothing may throw across the C ABI)
            shard();
        }
    }
    for (auto& t : threads) t.join();
    for (int k = 0; k < nctx; k++)
        if (rcs[(size_t)k] != PLAAC_OK && !(rcs[(size_t)k] == PLAAC_E_INVALID && hits)) return rcs[(size_t)k];
    int rc_shards = PLAAC_OK;
    for (int k = 0; k < nctx; k++)
        if (rcs[(size_t)k] != PLAAC_OK) rc_shards = rcs[(size_t)k];  // (invalid residue codes: reported after the merge)
    if (hits) {
        // The one exchange step of the path: every shard's candidate rows (its proteins with a CORE, or its top K) are
        // pulled onto the first GPU over NVLink (cudaMemcpyPeerAsync), ranked there as one set, and leave the box once.
        int64_t total = 0;
        for (int k = 0; k < nctx; k++)
            if (bounds[(size_t)k + 1] > bounds[(size_t)k]) {
                total += sh_hits[(size_t)k].count;
                hits->n_core += sh_hits[(size_t)k].n_core;
            }
        if (total > 0) {
            CU(c0, cudaSetDevice(c0->device));
            Slot& s0 = c0->slot[0];
            cudaStream_t st = s0.stream;
            int rc;
            if ((rc = ensure(c0, c0->union_rec, sizeof(plaac_summary) * (size_t)total))) return rc;
            if ((rc = ensure(c0, c0->union_idx, sizeof(int32_t) * (size_t)total))) return rc;
            if ((rc = ensure(c0, c0->union_order, sizeof(int32_t) * (size_t)total))) return rc;
            if ((rc = ensure(c0, c0->union_out_idx, sizeof(int32_t) * (size_t)total))) return rc;
            int64_t off = 0;
            for (int k = 0; k < nctx; k++) {
                const int64_t cnt = bounds[(size_t)k + 1] > bounds[(size_t)k] ? sh_hits[(size_t)k].count : 0;
                if (cnt <= 0) continue;
                const Slot& sk = ctxs[k]->slot[0];
                CU(c0, cudaMemcpyPeerAsync((plaac_summary*)c0->union_rec.p + off, c0->device, sk.summaries.p, ctxs[k]->device,
                                           sizeof(plaac_summary) * (size_t)cnt, st));
                CU(c0, cudaMemcpyPeerAsync((int32_t*)c0->union_idx.p + off, c0->device, sk.rk_order.p, ctxs[k]->device,
                                           sizeof(int32_t) * (size_t)cnt, st));
                k_hits_add_base<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>((int32_t*)c0->union_idx.p + off, cnt,
                                                                              (int32_t)bounds[(size_t)k]);
                c0->stats.kernel_launches += 1;
                off += cnt;
            }
            int64_t ncore_u = 0;
            if ((rc = plaac_rank_device(c0, (const plaac_summary*)c0->union_rec.p, total, 0, (int32_t*)c0->union_order.p, &ncore_u)))
                return rc;
            const int64_t want = hits->mode == PLAAC_HITS_CORE ? ncore_u : total;
            const int64_t count = std::min<int64_t>(hits->capacity, want);
            hits->count = count;
            if (count > 0) {
                if (!hits->records && !hits->index) return fail(c0, PLAAC_E_INVALID, "plaac_hits: no output array");
                if (hits->records) {
                    if ((rc = ensure(c0, s0.summaries, sizeof(plaac_summary) * (size_t)count))) return rc;
                    if ((rc = plaac_gather_device(c0, (const plaac_summary*)c0->union_rec.p, (const int32_t*)c0->union_order.p, count,
                                                  (plaac_summary*)s0.summaries.p)))
                        return rc;
                    if ((rc = d2h_any(c0, hits->records, s0.summaries.p, sizeof(plaac_summary) * (size_t)count, st))) return rc;
                }
                if (hits->index) {
                    k_hits_gather_idx<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(
                        (const int32_t*)c0->union_idx.p, (const int32_t*)c0->union_order.p, count, (int32_t*)c0->union_out_idx.p);
                    c0->stats.kernel_launches += 1;
                    if ((rc = d2h_any(c0, hits->index, c0->union_out_idx.p, sizeof(int32_t) * (size_t)count, st))) return rc;
                }
            }
            CU(c0, cudaStreamSynchronize(st));
            CU(c0, cudaGetLastError());
        }
    }
    return rc_shards;
} catch (...) {
    return api_caught((ctxs && nctx > 0 ? ctxs[0] : nullptr), "plaac_score_multi_packed");
}

}  // extern "C"

// The shuffle nulls on several ctxs (DESIGN.md section 15): every ctx scores every selected protein, each a range of
// its replicates.
namespace {

// Start of ctx c's part of a span of W replicates cut into n parts: floor(W c / n).
int64_t part_start(int64_t W, int c, int n) { return (int64_t)((__int128)W * c / n); }

// One phase of a multi-ctx call: rcs[c] = f(c) for every ctx c, one host thread each (the calling thread where no thread
// is to be had), all joined before it returns.  Returns the first non-zero code in ctx order.
template <class F>
int on_each_ctx(plaac_ctx* const* ctxs, int nctx, const char* fn, F f)
{
    std::vector<int> rcs((size_t)nctx, PLAAC_OK);
    std::vector<std::thread> threads;
    for (int c = 0; c < nctx; c++) {
        auto run = [&, c]() {
            try {
                rcs[(size_t)c] = f(c);
            } catch (...) {
                rcs[(size_t)c] = api_caught(ctxs[c], fn);
            }
        };
        try {
            threads.emplace_back(run);
        } catch (...) {
            run();
        }
    }
    for (auto& t : threads) t.join();
    for (int c = 0; c < nctx; c++)
        if (rcs[(size_t)c] != PLAAC_OK) return rcs[(size_t)c];
    return PLAAC_OK;
}

// Reference bytes > 21 seen by any ctx (its observed records or its replicates were scored in full all the same): the
// call returns PLAAC_E_INVALID at the end, with the text on ctxs[0], as the single call returns it.
struct BadBytes {
    std::mutex m;
    int rc = PLAAC_OK;
    std::string err;
    void note(int r, const std::string& e)
    {
        if (r != PLAAC_E_INVALID) return;
        std::lock_guard<std::mutex> g(m);
        rc = r;
        err = e;
    }
    int finish(plaac_ctx* c0)
    {
        if (rc != PLAAC_OK) c0->err = err;
        return rc;
    }
};

// Every ctx: null_observed over the whole selection (only ctxs[0] writes to the caller's observed).  Ctxs c >= 1 for
// which skip(c) holds score nothing and need no reference.
template <class Skip>
int multi_observed(plaac_ctx* const* ctxs, int nctx, const char* fn, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                   int64_t nsel, const int32_t* sel, int k, plaac_summary* observed, BadBytes& bad, Skip skip)
{
    return on_each_ctx(ctxs, nctx, fn, [&](int c) -> int {
        if (c > 0 && skip(c)) return PLAAC_OK;
        int rc_obs = PLAAC_OK;
        std::string err_obs;
        const int rc = null_observed(ctxs[c], codes, offsets, nprot, nsel, sel, k, c == 0 ? observed : nullptr, rc_obs, err_obs);
        bad.note(rc_obs, err_obs);
        return rc;
    });
}

}  // namespace

extern "C" {

int plaac_score_shuffles_multi(plaac_ctx* const* ctxs, int nctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                               plaac_null* null_spec, plaac_summary* observed)
try {
    const char* fn = "plaac_score_shuffles_multi";
    if (!ctxs || nctx < 1) return fail(nullptr, PLAAC_E_INVALID, "%s: no contexts", fn);
    for (int c = 0; c < nctx; c++)
        if (!ctxs[c]) return fail(nullptr, PLAAC_E_INVALID, "%s: NULL ctx %d", fn, c);
    if (nctx == 1) return plaac_score_shuffles(ctxs[0], codes, offsets, nprot, null_spec, observed);
    plaac_ctx* c0 = ctxs[0];
    if (!null_spec) return fail(c0, PLAAC_E_INVALID, "%s: NULL null_spec", fn);
    const plaac_null& N = *null_spec;
    const int64_t K = N.replicates;
    int64_t nsel = 0;
    const int32_t* sel = nullptr;
    int rc = null_check(c0, fn, nprot, N, nsel, sel);
    if (rc != PLAAC_OK || nsel == 0) return rc;
    const int k = __builtin_popcount((uint32_t)N.columns);
    const size_t ek = (size_t)k;
    BadBytes bad;
    auto r0 = [&](int c) { return part_start(K, c, nctx); };
    if ((rc = multi_observed(ctxs, nctx, fn, codes, offsets, nprot, nsel, sel, k, observed, bad,
                             [&](int c) { return r0(c + 1) == r0(c); })))
        return rc;
    // ctx c: replicates [r0(c), r0(c + 1)) of every selected protein, its counts and rows into host arrays of its own
    std::vector<std::vector<int64_t>> counts((size_t)nctx);
    rc = on_each_ctx(ctxs, nctx, fn, [&](int c) -> int {
        plaac_ctx* ctx = ctxs[c];
        const int64_t a = r0(c), W = r0(c + 1) - a;
        if (W == 0) return PLAAC_OK;
        std::vector<double> vals(N.values ? (size_t)nsel * (size_t)W * ek : 0);
        plaac_null R = N;
        R.replicates = W;
        R.nsel = nsel;
        R.proteins = sel;
        R.values = N.values ? vals.data() : nullptr;
        HostInput in;
        in.codes = codes;
        in.offsets = offsets;
        in.nref = nprot;
        in.nul = &R;
        in.r0 = a;
        int rc = score_host(ctx, in, nsel * W, nullptr, nullptr, nullptr);
        if (rc != PLAAC_OK && rc != PLAAC_E_INVALID) return rc;
        bad.note(rc, ctx->err);
        std::vector<int64_t>& cnt = counts[(size_t)c];
        cnt.resize((size_t)nsel * ek);
        cudaStream_t st = ctx->slot[0].stream;
        if ((rc = d2h_any(ctx, cnt.data(), ctx->null_counts.p, sizeof(int64_t) * cnt.size(), st))) return rc;
        CU(ctx, cudaStreamSynchronize(st));
        if (N.values)  // each protein's run of rows: j * K + a in the caller's array
            for (int64_t j = 0; j < nsel; j++)
                memcpy(N.values + ((size_t)j * (size_t)K + (size_t)a) * ek, vals.data() + (size_t)j * (size_t)W * ek,
                       sizeof(double) * (size_t)W * ek);
        return PLAAC_OK;
    });
    if (rc) return rc;
    for (size_t i = 0; i < (size_t)nsel * ek; i++) {
        int64_t sum = 0;
        for (const auto& cnt : counts)
            if (!cnt.empty()) sum += cnt[i];
        N.counts[i] = sum;
    }
    return bad.finish(c0);
} catch (...) {
    return api_caught((ctxs && nctx > 0 ? ctxs[0] : nullptr), "plaac_score_shuffles_multi");
}

// The rounds of plaac_score_shuffles_seq in lockstep on every ctx (DESIGN.md section 15).  Round g's span [R_{g-1}, R_g)
// is cut into one part per ctx; per slice of the active list (a sub-round, global over the ctxs): every ctx scores its
// part into hit flags relative to the part's start and counts each row's hits there (k_shuffle_stop with h above any
// count, over a zeroed table); the host walks each row's parts in ctx order from its count so far to the part where it
// reaches h; the ctxs holding such rows find their replicates (k_shuffle_stop with the base counts, h for the other rows,
// which it skips) and every ctx clears its flags.  count, L and the list live on the host.
int plaac_score_shuffles_seq_multi(plaac_ctx* const* ctxs, int nctx, const uint8_t* codes, const int64_t* offsets, int64_t nprot,
                                   const plaac_null* null_spec, int64_t stop_hits, int64_t* scored, plaac_summary* observed)
try {
    const char* fn = "plaac_score_shuffles_seq_multi";
    if (!ctxs || nctx < 1) return fail(nullptr, PLAAC_E_INVALID, "%s: no contexts", fn);
    for (int c = 0; c < nctx; c++)
        if (!ctxs[c]) return fail(nullptr, PLAAC_E_INVALID, "%s: NULL ctx %d", fn, c);
    if (nctx == 1) return plaac_score_shuffles_seq(ctxs[0], codes, offsets, nprot, null_spec, stop_hits, scored, observed);
    plaac_ctx* c0 = ctxs[0];
    int64_t nsel = 0;
    const int32_t* sel = nullptr;
    int rc = seq_check(c0, fn, nprot, null_spec, stop_hits, scored, nsel, sel);
    if (rc != PLAAC_OK || nsel == 0) return rc;
    const plaac_null& N = *null_spec;
    const int64_t K = N.replicates, h = stop_hits;
    const int k = __builtin_popcount((uint32_t)N.columns);
    const size_t ek = (size_t)k;
    BadBytes bad;
    if ((rc = multi_observed(ctxs, nctx, fn, codes, offsets, nprot, nsel, sel, k, observed, bad, [](int) { return false; })))
        return rc;
    // per ctx: seq_act[0] = the round's list, seq_act[1] = 0, 1, 2, ... (the rows of a slice: k_shuffle_stop then counts
    // and stops in tables of the slice's rows), null_counts = those tables, seq_scored and seq_live its other outputs
    std::vector<int32_t> iota((size_t)nsel);
    for (int64_t j = 0; j < nsel; j++) iota[(size_t)j] = (int32_t)j;
    rc = on_each_ctx(ctxs, nctx, fn, [&](int c) -> int {
        plaac_ctx* ctx = ctxs[c];
        cudaStream_t st = ctx->slot[0].stream;
        int rc;
        CU(ctx, cudaSetDevice(ctx->device));
        if ((rc = ensure(ctx, ctx->seq_scored, sizeof(int64_t) * (size_t)nsel * ek))) return rc;
        if ((rc = ensure(ctx, ctx->seq_live, sizeof(int32_t) * (size_t)nsel))) return rc;
        for (DevBuf& b : ctx->seq_act)
            if ((rc = ensure(ctx, b, sizeof(int32_t) * (size_t)(nsel + 1)))) return rc;
        if ((rc = h2d_any(ctx, ctx->seq_act[1].p, iota.data(), sizeof(int32_t) * (size_t)nsel, st))) return rc;
        // (a call that failed half-way may have left flags set)
        if (ctx->seq_flags.cap > 0) CU(ctx, cudaMemsetAsync(ctx->seq_flags.p, 0, ctx->seq_flags.cap, st));
        CU(ctx, cudaStreamSynchronize(st));
        return PLAAC_OK;
    });
    if (rc) return rc;

    // the schedule of section 14 with each part holding at least its ctx's chunk bound, and the tightest flag budget
    int64_t budget = INT64_MAX, chunk_res = 0;
    for (int c = 0; c < nctx; c++) {
        budget = std::min(budget, seq_budget(ctxs[c], k));
        chunk_res = std::max(chunk_res, ctxs[c]->chunk_res);
    }
    const int64_t wcap = budget / k * 32;
    std::vector<int64_t> count((size_t)nsel * ek, 0), L((size_t)nsel * ek, 0);
    std::vector<int32_t> act((size_t)nsel), ref((size_t)nsel), live((size_t)nsel);
    for (int64_t j = 0; j < nsel; j++) act[(size_t)j] = (int32_t)j;
    std::vector<int64_t> pa((size_t)nctx + 1);
    // per ctx, a row per (entry of the slice, column): its hits in the ctx's part, the base counts of step 3 and the L
    // it found
    std::vector<std::vector<int64_t>> hits((size_t)nctx), tab((size_t)nctx), at((size_t)nctx);
    std::vector<char> stops((size_t)nctx);
    int64_t nact = nsel, r0 = 0;
    while (nact > 0 && r0 < K) {
        int64_t res = 0;
        for (int64_t a = 0; a < nact; a++) {
            const int32_t j = act[(size_t)a];
            ref[(size_t)a] = sel ? sel[j] : j;
            res += offsets[ref[(size_t)a] + 1] - offsets[ref[(size_t)a]];
        }
        const int64_t W = seq_span(K, r0, h, nctx * seq_wmin(chunk_res, res), wcap), r1 = r0 + W;
        int64_t wpr_max = 0;
        for (int c = 0; c <= nctx; c++) pa[(size_t)c] = r0 + part_start(W, c, nctx);
        for (int c = 0; c < nctx; c++) wpr_max = std::max(wpr_max, (pa[(size_t)c + 1] - pa[(size_t)c] + 31) / 32);
        const int64_t per = std::max<int64_t>(1, budget / (k * wpr_max));  // entries per sub-round
        std::fill(live.begin(), live.begin() + nact, 0);
        for (int64_t a0 = 0; a0 < nact; a0 += per) {
            const int64_t n = std::min(per, nact - a0), rows = n * k;
            // 1. every ctx scores its part of the slice and counts each row's hits there
            rc = on_each_ctx(ctxs, nctx, fn, [&](int c) -> int {
                plaac_ctx* ctx = ctxs[c];
                const int64_t p0 = pa[(size_t)c], p1 = pa[(size_t)c + 1], wpr = (p1 - p0 + 31) / 32;
                hits[(size_t)c].assign((size_t)rows, 0);
                if (p1 == p0) return PLAAC_OK;
                cudaStream_t st = ctx->slot[0].stream;
                int rc;
                CU(ctx, cudaSetDevice(ctx->device));
                if (a0 == 0) CU(ctx, cudaMemcpyAsync(ctx->seq_act[0].p, act.data(), sizeof(int32_t) * (size_t)nact, cudaMemcpyHostToDevice, st));
                const size_t cap0 = ctx->seq_flags.cap;
                if ((rc = ensure(ctx, ctx->seq_flags, sizeof(uint32_t) * (size_t)(rows * wpr)))) return rc;
                if (ctx->seq_flags.cap != cap0) CU(ctx, cudaMemsetAsync(ctx->seq_flags.p, 0, ctx->seq_flags.cap, st));
                CU(ctx, cudaStreamSynchronize(st));  // (the chunks run on the other slots' streams too)
                const SeqRound sr = {(const int32_t*)ctx->seq_act[0].p + a0, (uint32_t*)ctx->seq_flags.p, wpr};
                plaac_null R = N;
                R.replicates = p1 - p0;
                R.nsel = n;
                R.proteins = ref.data() + a0;
                R.counts = nullptr;
                R.values = nullptr;
                HostInput in;
                in.codes = codes;
                in.offsets = offsets;
                in.nref = nprot;
                in.nul = &R;
                in.r0 = p0;
                in.seq = &sr;
                rc = score_host(ctx, in, n * (p1 - p0), nullptr, nullptr, nullptr);  // (returns with every slot synchronised)
                if (rc != PLAAC_OK && rc != PLAAC_E_INVALID) return rc;
                bad.note(rc, ctx->err);
                int64_t* d_tab = (int64_t*)ctx->null_counts.p;
                CU(ctx, cudaMemsetAsync(d_tab, 0, sizeof(int64_t) * (size_t)rows, st));
                k_shuffle_stop<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(sr.flags, (const int32_t*)ctx->seq_act[1].p, n, k, wpr,
                                                                           INT64_MAX, p0, p1, K, d_tab, (int64_t*)ctx->seq_scored.p,
                                                                           (int32_t*)ctx->seq_live.p);
                ctx->stats.kernel_launches += 1;
                CU(ctx, cudaMemcpyAsync(hits[(size_t)c].data(), d_tab, sizeof(int64_t) * (size_t)rows, cudaMemcpyDeviceToHost, st));
                CU(ctx, cudaStreamSynchronize(st));
                return PLAAC_OK;
            });
            if (rc) return rc;
            // 2. each row's parts in ctx order, from its count so far
            std::fill(stops.begin(), stops.end(), 0);
            for (int c = 0; c < nctx; c++) tab[(size_t)c].assign((size_t)rows, h);
            for (int64_t row = 0; row < rows; row++) {
                const int64_t a = a0 + row / k, s = (int64_t)act[(size_t)a] * k + row % k;
                int64_t n_hit = count[(size_t)s];
                if (n_hit >= h) continue;  // stopped in an earlier round
                int c = 0;
                for (; c < nctx; c++) {
                    const int64_t x = hits[(size_t)c][(size_t)row];
                    if (n_hit + x >= h) break;
                    n_hit += x;
                }
                if (c < nctx) {
                    tab[(size_t)c][(size_t)row] = n_hit;
                    stops[(size_t)c] = 1;
                    count[(size_t)s] = h;
                } else {
                    count[(size_t)s] = n_hit;
                    L[(size_t)s] = r1;
                    if (r1 < K) live[(size_t)a] = 1;
                }
            }
            // 3. the ctxs holding stopping rows find their replicates; every ctx clears its flags
            rc = on_each_ctx(ctxs, nctx, fn, [&](int c) -> int {
                plaac_ctx* ctx = ctxs[c];
                const int64_t p0 = pa[(size_t)c], p1 = pa[(size_t)c + 1], wpr = (p1 - p0 + 31) / 32;
                if (p1 == p0) return PLAAC_OK;
                cudaStream_t st = ctx->slot[0].stream;
                CU(ctx, cudaSetDevice(ctx->device));
                if (stops[(size_t)c]) {
                    int64_t* d_tab = (int64_t*)ctx->null_counts.p;
                    CU(ctx, cudaMemcpyAsync(d_tab, tab[(size_t)c].data(), sizeof(int64_t) * (size_t)rows, cudaMemcpyHostToDevice, st));
                    k_shuffle_stop<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>((const uint32_t*)ctx->seq_flags.p,
                                                                               (const int32_t*)ctx->seq_act[1].p, n, k, wpr, h, p0, p1,
                                                                               K, d_tab, (int64_t*)ctx->seq_scored.p,
                                                                               (int32_t*)ctx->seq_live.p);
                    ctx->stats.kernel_launches += 1;
                    at[(size_t)c].resize((size_t)rows);
                    CU(ctx, cudaMemcpyAsync(at[(size_t)c].data(), ctx->seq_scored.p, sizeof(int64_t) * (size_t)rows,
                                            cudaMemcpyDeviceToHost, st));
                }
                CU(ctx, cudaMemsetAsync(ctx->seq_flags.p, 0, sizeof(uint32_t) * (size_t)(rows * wpr), st));
                CU(ctx, cudaStreamSynchronize(st));
                return PLAAC_OK;
            });
            if (rc) return rc;
            for (int c = 0; c < nctx; c++)
                if (stops[(size_t)c])
                    for (int64_t row = 0; row < rows; row++)
                        if (tab[(size_t)c][(size_t)row] < h)
                            L[(size_t)act[(size_t)(a0 + row / k)] * ek + (size_t)(row % k)] = at[(size_t)c][(size_t)row];
        }
        // the next round's list: the entries with a column below h, in list order
        int64_t m = 0;
        for (int64_t a = 0; a < nact; a++)
            if (live[(size_t)a]) act[(size_t)m++] = act[(size_t)a];
        nact = m;
        r0 = r1;
    }
    memcpy(N.counts, count.data(), sizeof(int64_t) * count.size());
    memcpy(scored, L.data(), sizeof(int64_t) * L.size());
    return bad.finish(c0);
} catch (...) {
    return api_caught((ctxs && nctx > 0 ? ctxs[0] : nullptr), "plaac_score_shuffles_seq_multi");
}

}  // extern "C"


// ------------------------------------------------------------------------------------------------ FASTA ingest
extern "C" {

int plaac_ingest_fasta_device(plaac_ctx* ctx, const char* d_text, int64_t nbytes, uint8_t* d_codes, int64_t* d_offsets,
                              int64_t* d_name_pos, int32_t* d_name_len, uint8_t* d_flags, int64_t max_rec,
                              plaac_fasta_index* index, uint64_t* d_bg_counts)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_ingest_fasta_device: NULL ctx");
    if (nbytes < 0 || max_rec < 0 || !index) return fail(ctx, PLAAC_E_INVALID, "bad size / NULL index");
    if (nbytes > 0 && (!d_text || !d_codes)) return fail(ctx, PLAAC_E_INVALID, "NULL text/codes");
    if (!d_offsets) return fail(ctx, PLAAC_E_INVALID, "NULL offsets");
    CU(ctx, cudaSetDevice(ctx->device));
    Slot& s = ctx->slot[0];
    cudaStream_t st = s.stream;
    index->nrec = index->nres = 0;
    const long long ntiles = (nbytes + kIngTile - 1) / kIngTile;
    int rc;
    if ((rc = ensure(ctx, s.ing_agg, sizeof(Ing3) * (size_t)std::max<long long>(ntiles, 1)))) return rc;
    if ((rc = ensure(ctx, s.ing_cnt, sizeof(int32_t) * (size_t)std::max<long long>(ntiles, 1)))) return rc;
    if ((rc = ensure(ctx, s.ing_base, sizeof(int64_t) * (size_t)(ntiles + 1)))) return rc;
    if ((rc = ensure(ctx, s.ing_misc, sizeof(Ing3) + 64))) return rc;
    // flags are OR-ed into: zero them (rounded up to whole words); also used internally when the caller passes NULL
    uint8_t* flags = d_flags;
    int64_t* npos = d_name_pos;
    int32_t* nlen = d_name_len;
    const size_t cap = (size_t)std::max<int64_t>(max_rec, 1);
    if (!flags) {
        if ((rc = ensure(ctx, s.ing_flags, cap + 8))) return rc;
        flags = (uint8_t*)s.ing_flags.p;
    }
    if (!npos) {
        if ((rc = ensure(ctx, s.ing_npos, sizeof(int64_t) * cap))) return rc;
        npos = (int64_t*)s.ing_npos.p;
    }
    if (!nlen) {
        if ((rc = ensure(ctx, s.ing_nlen, sizeof(int32_t) * cap))) return rc;
        nlen = (int32_t*)s.ing_nlen.p;
    }
    if (((uintptr_t)flags & 3) != 0) return fail(ctx, PLAAC_E_INVALID, "flags must be 4-byte aligned");
    CU(ctx, cudaMemsetAsync(flags, 0, (size_t)max_rec, st));
    Ing3 grand;
    grand.ls = grand.mk = -1;
    grand.nh = 0;
    long long total = 0;
    if (ntiles > 0) {
        const unsigned char* t = (const unsigned char*)d_text;
        k_ing_reduce<<<(unsigned)ntiles, kIngThreads, 0, st>>>(t, nbytes, (Ing3*)s.ing_agg.p);
        k_ing_scan3<<<1, 1024, 0, st>>>((Ing3*)s.ing_agg.p, ntiles, (Ing3*)s.ing_misc.p);
        IngOut out;
        out.codes = d_codes;
        out.offsets = (long long*)d_offsets;
        out.name_pos = (long long*)npos;
        out.name_len = nlen;
        out.flags = flags;
        out.max_rec = max_rec;
        k_ing_apply<0><<<(unsigned)ntiles, kIngThreads, 0, st>>>(t, nbytes, (const Ing3*)s.ing_agg.p, (int32_t*)s.ing_cnt.p,
                                                                  nullptr, out);
        k_scan_exclusive<int32_t><<<1, 1024, 0, st>>>((const int32_t*)s.ing_cnt.p, (int64_t*)s.ing_base.p, ntiles);
        k_ing_apply<1><<<(unsigned)ntiles, kIngThreads, 0, st>>>(t, nbytes, (const Ing3*)s.ing_agg.p, nullptr,
                                                                  (const long long*)s.ing_base.p, out);
        ctx->stats.kernel_launches += 5;
        CU(ctx, cudaMemcpyAsync(&grand, s.ing_misc.p, sizeof(Ing3), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(&total, (int64_t*)s.ing_base.p + ntiles, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
    }
    index->nrec = grand.nh;
    index->nres = total;
    const int64_t stored = std::min<int64_t>(grand.nh, max_rec);
    // closing offset of the last stored record
    if (stored == grand.nh) {
        CU(ctx, cudaMemcpyAsync(d_offsets + stored, &total, sizeof(int64_t), cudaMemcpyHostToDevice, st));
    } else {
        // truncated: record `stored` exists in the text; its start is the end of the last stored one.  Re-deriving
        // it would need its header; report the truncation instead.
        return fail(ctx, PLAAC_E_INVALID, "FASTA holds %lld records but max_rec is %lld", (long long)grand.nh,
                    (long long)max_rec);
    }
    if (d_bg_counts) {
        CU(ctx, cudaMemsetAsync(d_bg_counts, 0, sizeof(uint64_t) * PLAAC_NAA, st));
        if (stored > 0) {
            const unsigned grid = (unsigned)std::min<int64_t>((stored + 7) / 8, (int64_t)ctx->sm_count * 8);
            k_bg_hist<<<grid, 256, 0, st>>>(d_codes, (const long long*)d_offsets, flags, stored,
                                            (unsigned long long*)d_bg_counts);
            ctx->stats.kernel_launches += 1;
        }
    }
    CU(ctx, cudaStreamSynchronize(st));
    CU(ctx, cudaGetLastError());
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_ingest_fasta_device");
}

int plaac_ingest_fasta(plaac_ctx* ctx, const char* text, int64_t nbytes, uint8_t* codes, int64_t* offsets, int64_t* name_pos,
                       int32_t* name_len, uint8_t* flags, int64_t max_rec, plaac_fasta_index* index, double* bg_counts)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_ingest_fasta: NULL ctx");
    if (nbytes < 0 || max_rec < 0 || !index || !offsets) return fail(ctx, PLAAC_E_INVALID, "bad size / NULL argument");
    if (nbytes > 0 && (!text || !codes)) return fail(ctx, PLAAC_E_INVALID, "NULL text/codes");
    CU(ctx, cudaSetDevice(ctx->device));
    Slot& s = ctx->slot[0];
    int rc;
    const size_t cap = (size_t)std::max<int64_t>(max_rec, 1);
    if ((rc = ensure(ctx, s.ing_text, (size_t)nbytes + 64))) return rc;
    if ((rc = ensure(ctx, s.ing_codes, (size_t)nbytes + 64))) return rc;
    if ((rc = ensure(ctx, s.ing_offsets, sizeof(int64_t) * (cap + 1)))) return rc;
    if ((rc = ensure(ctx, s.ing_npos, sizeof(int64_t) * cap))) return rc;
    if ((rc = ensure(ctx, s.ing_nlen, sizeof(int32_t) * cap))) return rc;
    if ((rc = ensure(ctx, s.ing_flags, cap + 8))) return rc;
    if ((rc = ensure(ctx, s.ing_hist, sizeof(uint64_t) * PLAAC_NAA))) return rc;
    if (nbytes > 0) CU(ctx, cudaMemcpyAsync(s.ing_text.p, text, (size_t)nbytes, cudaMemcpyHostToDevice, s.stream));
    rc = plaac_ingest_fasta_device(ctx, (const char*)s.ing_text.p, nbytes, (uint8_t*)s.ing_codes.p, (int64_t*)s.ing_offsets.p,
                                   (int64_t*)s.ing_npos.p, (int32_t*)s.ing_nlen.p, (uint8_t*)s.ing_flags.p, max_rec, index,
                                   bg_counts ? (uint64_t*)s.ing_hist.p : nullptr);
    if (rc != PLAAC_OK) return rc;
    const size_t nrec = (size_t)index->nrec;
    if (index->nres > 0) CU(ctx, cudaMemcpy(codes, s.ing_codes.p, (size_t)index->nres, cudaMemcpyDeviceToHost));
    CU(ctx, cudaMemcpy(offsets, s.ing_offsets.p, sizeof(int64_t) * (nrec + 1), cudaMemcpyDeviceToHost));
    if (name_pos && nrec) CU(ctx, cudaMemcpy(name_pos, s.ing_npos.p, sizeof(int64_t) * nrec, cudaMemcpyDeviceToHost));
    if (name_len && nrec) CU(ctx, cudaMemcpy(name_len, s.ing_nlen.p, sizeof(int32_t) * nrec, cudaMemcpyDeviceToHost));
    if (flags && nrec) CU(ctx, cudaMemcpy(flags, s.ing_flags.p, nrec, cudaMemcpyDeviceToHost));
    if (bg_counts) {
        uint64_t h[PLAAC_NAA];
        CU(ctx, cudaMemcpy(h, s.ing_hist.p, sizeof(h), cudaMemcpyDeviceToHost));
        for (int i = 0; i < PLAAC_NAA; i++) bg_counts[i] = (double)h[i];
    }
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_ingest_fasta");
}

}  // extern "C"


extern "C" int plaac_score_fasta(plaac_ctx* ctx, const char* text, int64_t nbytes, int64_t max_rec, plaac_summary* summaries,
                                 uint8_t* codes, int64_t* offsets, int64_t* name_pos, int32_t* name_len, uint8_t* flags,
                                 plaac_fasta_index* index, double* bg_counts)
try {
    if (!ctx) return fail(nullptr, PLAAC_E_INVALID, "plaac_score_fasta: NULL ctx");
    if (nbytes < 0 || max_rec < 0 || !index || !offsets || !summaries) return fail(ctx, PLAAC_E_INVALID, "bad size / NULL argument");
    if (nbytes > 0 && !text) return fail(ctx, PLAAC_E_INVALID, "NULL text");
    CU(ctx, cudaSetDevice(ctx->device));
    Slot& s = ctx->slot[0];
    int rc;
    const size_t cap = (size_t)std::max<int64_t>(max_rec, 1);
    if ((rc = ensure(ctx, s.ing_text, (size_t)nbytes + 64))) return rc;
    if ((rc = ensure(ctx, s.ing_codes, (size_t)nbytes + 64))) return rc;
    if ((rc = ensure(ctx, s.ing_offsets, sizeof(int64_t) * (cap + 1)))) return rc;
    if ((rc = ensure(ctx, s.ing_npos, sizeof(int64_t) * cap))) return rc;
    if ((rc = ensure(ctx, s.ing_nlen, sizeof(int32_t) * cap))) return rc;
    if ((rc = ensure(ctx, s.ing_flags, cap + 8))) return rc;
    if ((rc = ensure(ctx, s.ing_hist, sizeof(uint64_t) * PLAAC_NAA))) return rc;
    if ((rc = h2d_any(ctx, s.ing_text.p, text, (size_t)nbytes, s.stream))) return rc;
    rc = plaac_ingest_fasta_device(ctx, (const char*)s.ing_text.p, nbytes, (uint8_t*)s.ing_codes.p, (int64_t*)s.ing_offsets.p,
                                   (int64_t*)s.ing_npos.p, (int32_t*)s.ing_nlen.p, (uint8_t*)s.ing_flags.p, max_rec, index,
                                   bg_counts ? (uint64_t*)s.ing_hist.p : nullptr);
    if (rc != PLAAC_OK) return rc;
    const size_t nrec = (size_t)index->nrec;
    if (nrec > 0) {
        if ((rc = ensure(ctx, s.summaries, sizeof(plaac_summary) * nrec))) return rc;
        rc = plaac_score_device(ctx, (const uint8_t*)s.ing_codes.p, (const int64_t*)s.ing_offsets.p, (int64_t)nrec, index->nres,
                                (plaac_summary*)s.summaries.p, nullptr);
        if (rc != PLAAC_OK) return rc;
        // the index arrays travel back while the scoring kernels run (pageable destinations through the staging buffers)
        cudaStream_t cp = s.aux1;
        if (codes && (rc = d2h_any(ctx, codes, s.ing_codes.p, (size_t)index->nres, cp))) return rc;
        if ((rc = d2h_any(ctx, offsets, s.ing_offsets.p, sizeof(int64_t) * (nrec + 1), cp))) return rc;
        if (name_pos && (rc = d2h_any(ctx, name_pos, s.ing_npos.p, sizeof(int64_t) * nrec, cp))) return rc;
        if (name_len && (rc = d2h_any(ctx, name_len, s.ing_nlen.p, sizeof(int32_t) * nrec, cp))) return rc;
        if (flags && (rc = d2h_any(ctx, flags, s.ing_flags.p, nrec, cp))) return rc;
        if ((rc = d2h_any(ctx, summaries, s.summaries.p, sizeof(plaac_summary) * nrec, s.stream))) return rc;
        rc = plaac_sync(ctx);
        CU(ctx, cudaStreamSynchronize(cp));
        if (rc != PLAAC_OK) return rc;
    } else {
        CU(ctx, cudaMemcpy(offsets, s.ing_offsets.p, sizeof(int64_t), cudaMemcpyDeviceToHost));
    }
    if (bg_counts) {
        uint64_t h[PLAAC_NAA];
        CU(ctx, cudaMemcpy(h, s.ing_hist.p, sizeof(h), cudaMemcpyDeviceToHost));
        for (int i = 0; i < PLAAC_NAA; i++) bg_counts[i] = (double)h[i];
    }
    return PLAAC_OK;
} catch (...) {
    return api_caught(ctx, "plaac_score_fasta");
}


