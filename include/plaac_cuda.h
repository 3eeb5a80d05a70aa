/*
 * plaac_cuda.h -- C ABI of libplaac_cuda.so: the B200 (sm_100a) implementation
 * of PLAAC's per-protein scoring hot path.
 *
 * The reference (whitehead/plaac, cli/src/plaac.java; "plaac.java:N" below) has
 * no FFI seam: the path is reached by plain Java calls from the two driver
 * loops scoreallfastas (plaac.java:755-948) and plotsomefastas (:610-647).
 * This header is the seam a host (Java via java.lang.foreign / JNI, C++, or
 * Python ctypes) binds instead of those calls; INTEGRATION.md shows the stubs.
 *
 * Conventions
 *  - plain C symbols, plain pointers and sizes; no C++/torch types;
 *  - every function returns 0 on success or a negative PLAAC_E_* code and
 *    never throws/aborts across the ABI; plaac_last_error() has the text;
 *  - the caller owns every buffer it passes; the library owns device memory;
 *  - a ctx is bound to ONE GPU and used by one host thread at a time
 *    (multi-GPU = one ctx + one thread/process per GPU; proteins are
 *    independent, no collective is needed);
 *  - results are written in input order;
 *  - positions are 0-based exactly as plaac.java holds them internally; the
 *    host adds 1 when printing (plaac.java:899-945).
 *  - the host computes every table with its own Math.log/exp (plaac.java:279-299,
 *    :449-500, :968-1001, :2893-2935); the device only does IEEE double
 *    + - * / floor compare (no FMA contraction), so reference-order results are
 *    reproducible bit for bit where the algorithm is evaluated in reference order.
 */
#ifndef PLAAC_CUDA_H
#define PLAAC_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLAAC_NAA 22        /* plaac.java:26  X A C D E F G H I K L M N P Q R S T V W Y *  */
#define PLAAC_LUT_LEN 4001  /* plaac.java:34,282  loglut[0..4000] */

#define PLAAC_OK 0
#define PLAAC_E_INVALID (-1)     /* bad argument (NULL, negative size, offsets not monotone, code > 21) */
#define PLAAC_E_CUDA (-2)        /* CUDA runtime error (text in plaac_last_error) */
#define PLAAC_E_UNSUPPORTED (-3) /* parameter combination outside what the kernels implement */
#define PLAAC_E_NOMEM (-4)       /* device or pinned-host allocation failed */
#define PLAAC_E_NODEVICE (-5)    /* no CUDA device / not an sm_100 device */

/* Everything scoreallfastas/plotsomefastas receive from main (plaac.java:526-528)
 * plus the static tables of class plaac, already in log space. */
typedef struct plaac_params {
    int32_t core_len;        /* -c, plaac.java:317 (default 60) */
    int32_t ww1;             /* -w FoldIndex window, :318 (41) */
    int32_t ww2;             /* -W PAPA window, :319 (41) */
    int32_t ww3;             /* PLAAC-LLR smoothing window, :320,:355 (= ww2) */
                             /* (ww1, ww2, ww3 are independent as in the jar; settings whose half-widths differ take
                                tap-by-tap kernels in the jar's operation order instead of the streaming ones) */
    int32_t adjust_prolines; /* :328 (1) */
    int32_t mw_window;       /* :767 (80) */
    int32_t reserved[2];
    /* hmm1 = prionhmm1(fg,bg), :968-981, after hmm.initialize :2893-2935 */
    double lt[2][2];         /* ltprob[from][to] */
    double li[2];            /* liprob */
    double lf[2];            /* lfprob (0,0 for PLAAC's models) */
    double le[2][PLAAC_NAA]; /* leprob[state][aa]; state 0 = background, 1 = PrD-like */
    /* hmm0 = prionhmm0(bg), :988-1001: identity transitions, starts in state 0,
     * so its Viterbi and marginal log-probabilities are both the sequential sum
     * of le0[aa_t] (SURVEY.md section 8 a5). */
    double le0[PLAAC_NAA];
    double llr[PLAAC_NAA];      /* :497-500 */
    double papa_lod[PLAAC_NAA]; /* lodpapa1, :285-291 */
    double hydro2[PLAAC_NAA];   /* aahydro2, :90 */
    double charge[PLAAC_NAA];   /* aacharge, :37-60 (must be small integers) */
    double fi_cc[3];            /* {2.785, -1, -1.151}, :800 */
    double big_neg;             /* -1e6, :817 */
    double ln2;                 /* Math.log(2), :30 */
    double loglut[PLAAC_LUT_LEN]; /* :282-283 */
} plaac_params;

/* One row of the summary table (plaac.java:899-945) before formatting:
 * 14 x int32 + 13 x double = 160 bytes, no padding. */
typedef struct plaac_summary {
    int32_t mw_score, mw_start, mw_end;               /* hs1, :771 */
    int32_t llr_start, llr_end;                       /* hs2, :783; -1/-2 when PROTlen < c */
    int32_t vit_maxrun;                               /* longestrun(viterbipath), :814 */
    int32_t core_start, core_end, prd_start, prd_end; /* :851-880; -1/-2 when no CORE */
    int32_t prot_len;                                 /* 0 => the jar prints no row (:762) */
    int32_t fi_numaa, fi_maxrun;                      /* numdisorderedstrict2, maxlen :5010-5060 */
    int32_t papa_center;                              /* papamaxcenter (-1 if none), :4941-4948 */
    double llr;          /* hs2[2]; -Inf when PROTlen < c (host prints NaN via inf2nan) */
    double core_score;   /* hs3[2] or NaN */
    double prd_score;    /* 0.0 when no CORE */
    double hmm_all;      /* hmm1.lmarginalprob - hmm0.lmarginalprob, :797 */
    double hmm_vit;      /* hmm1.lviterbiprob - hmm0.lviterbiprob, :798 */
    double fi_meanhydro, fi_meancharge, fi_meancombo; /* :4876-4883 */
    double papa_combo;   /* papamaxscore (-Inf if none), :4931 */
    double papa_prop, papa_fi, papa_llr, papa_llr2;   /* :4990-4996 (NaN if none) */
} plaac_summary;

/* Per-residue table (plaac.java:603-605, :637-641), struct of arrays, each array
 * as long as the total residue count of the call; element offsets[i]+t belongs to
 * residue t of protein i.  82 bytes per residue. */
typedef struct plaac_residue_out {
    uint8_t *vit, *map;
    double *charge, *hydro, *fi, *plaac, *papa, *fix2, *plaacx2, *papax2;
    double *post_bg, *post_prd;
} plaac_residue_out;

typedef struct plaac_ctx plaac_ctx; /* opaque */

int plaac_device_count(void);

/* Validates params, uploads the tables, creates the stream.  Replaces the
 * construction of hmm1/hmm0 + static tables for the device side. */
int plaac_create(plaac_ctx **out, int device, const plaac_params *params);
void plaac_destroy(plaac_ctx *ctx);

/* Text of the last error on this ctx (ctx == NULL: last error of plaac_create /
 * plaac_device_count on the calling thread).  Never NULL. */
const char *plaac_last_error(const plaac_ctx *ctx);

/* Summary mode and (per_res != NULL) per-residue mode with HOST buffers:
 * replaces the bodies of plaac.java:755-948 / :610-647 for a batch.
 *   codes    1 byte per residue, 0..21 (aatoint :1508-1534), terminal '*' already
 *            stripped (:758); proteins concatenated;
 *   offsets  nprot+1 monotone int64; protein i = codes[offsets[i] .. offsets[i+1])
 *   summaries nprot records (may be NULL if per_res != NULL)
 *   per_res  NULL, or host arrays offsets[nprot]-offsets[0] long.
 * Input is processed in device-sized chunks, copies overlapped with compute;
 * pinned host buffers make the copies asynchronous.  Blocks until done. */
int plaac_score(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                plaac_summary *summaries, const plaac_residue_out *per_res);

/* Page-locked host memory for the buffers handed to plaac_score / plaac_score_multi / plaac_ingest_fasta.  The
 * reference has no counterpart (its arrays live on the Java heap, plaac.java:755-948); a host that keeps the batch in
 * ordinary pageable memory still gets correct results, but the driver then stages every copy and the chunk pipeline of
 * plaac_score runs at a fraction of the PCIe rate (DESIGN.md section 7).  Usable before any ctx exists; errors are
 * reported like plaac_create's (plaac_last_error(NULL)).
 *   plaac_host_alloc     new pinned block (flags: 0, or PLAAC_HOST_WRITE_COMBINED for blocks the host only writes
 *                        sequentially, e.g. codes: not cached on the CPU side, slow to read back);
 *   plaac_host_register  pins memory the host already owns (a Java FFM MemorySegment, a malloc'd block); pinning costs
 *                        about as much as one pass over the memory, so register buffers that are reused. */
#define PLAAC_HOST_WRITE_COMBINED 1
int plaac_host_alloc(void **out, size_t bytes, int flags);
int plaac_host_free(void *p);
int plaac_host_register(void *p, size_t bytes);
int plaac_host_unregister(void *p);

/* Same with DEVICE buffers already resident on ctx's GPU (offsets[0] must be 0,
 * ntotal = offsets[nprot]).  Work is enqueued on the ctx stream; call
 * plaac_sync() (or synchronise plaac_stream()) before reading the outputs. */
int plaac_score_device(plaac_ctx *ctx, const uint8_t *d_codes, const int64_t *d_offsets, int64_t nprot,
                       int64_t ntotal, plaac_summary *d_summaries, const plaac_residue_out *d_per_res);
int plaac_sync(plaac_ctx *ctx);
void *plaac_stream(plaac_ctx *ctx); /* cudaStream_t of the ctx */

/* ---- transport-lean batch call -----------------------------------------------------------------------------
 * Same scoring as plaac_score() with fewer bytes on the host link, which is what bounds the host-buffer call
 * (DESIGN.md section 7).  The reference has no counterpart: its arrays never leave the Java heap (plaac.java:755-948).
 *
 *   IN   residues as radix-22 words: 7 residue codes per uint32, word = c0 + 22*c1 + ... + 22^6*c6 (22^7 < 2^32),
 *        i.e. 4/7 = 0.571 byte per residue instead of 1; the batch's residues are concatenated WITHOUT regard to
 *        protein boundaries (residue r of the batch is digit r%7 of word r/7; unused digits of the last word are 0);
 *        int32 lengths instead of int64 offsets.
 *   OUT  optionally not the whole table but its head in the order the reference's consumer gives it
 *        (web/lib/server.rb:222-229, "TODO: move this sorting into the java"): every protein with a CORE, or the top K
 *        rows, best first, each with the index of its protein in the batch. */
#define PLAAC_PACK_PER_WORD 7
/* number of uint32 words that hold nres residues: ceil(nres / 7) */
int64_t plaac_packed_words(int64_t nres);
/* codes (0..21, one byte each; larger bytes are packed as X and the call returns PLAAC_E_INVALID after packing
 * everything) -> words.  nthreads <= 0: all host threads.  Pure host code (no GPU, no ctx). */
int plaac_pack_host(const uint8_t *codes, int64_t nres, uint32_t *words, int nthreads);
/* The same for a batch that is built piece by piece: packs codes[0 .. nres) at residue positions [pos, pos + nres) of
 * the batch.  The word that holds residue pos keeps its digits below pos % 7; pieces must be appended in order. */
int plaac_pack_append_host(const uint8_t *codes, int64_t nres, uint32_t *words, int64_t pos, int nthreads);
/* FASTA letters -> words in one pass: aatoint (plaac.java:1508-1534) fused with the packing. */
int plaac_pack_chars_host(const char *chars, int64_t nres, uint32_t *words, int nthreads);
/* words -> codes for residues [first, first + count) of the packed batch (the host needs residues again for the
 * string columns COREaa .. PAPAaa, plaac.java:915-944). */
int plaac_unpack_host(const uint32_t *words, int64_t first, int64_t count, uint8_t *codes);

#define PLAAC_HITS_CORE 1 /* every protein with a CORE (COREscore not NaN), ranked */
#define PLAAC_HITS_TOPK 2 /* the first `capacity` rows of the ranking of the whole batch */
typedef struct plaac_hits {
    int32_t mode;           /* in: PLAAC_HITS_CORE or PLAAC_HITS_TOPK */
    int32_t rank_flags;     /* in: reserved, must be 0 */
    int64_t capacity;       /* in: rows `records` and `index` can hold */
    plaac_summary *records; /* out: `count` rows, best first (COREscore desc, LLR desc, input order) */
    int32_t *index;         /* out: index of each row's protein in the batch */
    int64_t count;          /* out: rows written = min(capacity, rows the mode selects) */
    int64_t n_core;         /* out: proteins of the batch with a CORE (may exceed capacity) */
} plaac_hits;

/* words/lengths as above, nres = sum of lengths (checked).  summaries: nprot records in input order, or NULL when only
 * hits are wanted; hits: NULL or the compact output (at least one of the two).  per_res as in plaac_score (element
 * index = residue index in the batch).  HOST buffers, pinned or not, chunked and pipelined exactly like plaac_score;
 * records are bit-identical to plaac_score's.  nprot < 2^31 when hits are requested. */
int plaac_score_packed(plaac_ctx *ctx, const uint32_t *words, const int32_t *lengths, int64_t nprot, int64_t nres,
                       plaac_summary *summaries, const plaac_residue_out *per_res, plaac_hits *hits);
/* The same compact output for the one-byte codes of plaac_score(). */
int plaac_score_hits(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot, plaac_hits *hits);

/* ---- sequence variants (DESIGN.md section 11): substitution lists expanded on the device --------------------------
 * Variants of the proteins of a reference batch: variant v is protein protein[v] with the residues at
 * pos[first_sub[v] .. first_sub[v+1]) replaced by code[...] (0-based positions, strictly increasing within a variant;
 * a variant with no substitution is the wild type). */
typedef struct plaac_variants {
    int64_t nvar;
    const int32_t *protein;    /* nvar indices into the reference batch */
    const int64_t *first_sub;  /* nvar + 1, first_sub[0] == 0, non-decreasing */
    const int32_t *pos;        /* first_sub[nvar] positions, each < the protein's length */
    const uint8_t *code;       /* first_sub[nvar] new residue codes, 0..21 */
} plaac_variants;

/* codes/offsets/nprot: the reference batch, exactly as plaac_score takes it (HOST buffers).  summaries: nvar records in
 * variant order, each byte-identical to plaac_score's record for the mutated protein.  Blocks until done.  Summary mode
 * only.  The reference is uploaded once; per chunk of the variant list only its slice of the four arrays crosses the
 * link, and the variant residues are built on the device.
 * PLAAC_E_INVALID, with the variant's index in plaac_last_error: a protein index outside [0, nprot), a position outside
 * the protein, positions of a variant that do not strictly increase, a code > 21, a bad first_sub array, or a NULL array
 * with nvar > 0.  The substitutions are validated during the chunk walk, so the records of earlier chunks may already
 * have been written when such an error is returned.  nvar == 0: PLAAC_OK, nothing written.  Reference bytes > 21 are
 * scored as X and reported as PLAAC_E_INVALID after the batch, as in plaac_score.  The call's chunks use the automatic
 * long-path threshold (plaac_set_long_path(ctx, -1, .)) whatever the ctx's setting, which it leaves unchanged: records do
 * not depend on the threshold, and equal-length variants are scored most efficiently by the bucketed kernel. */
int plaac_score_variants(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                         const plaac_variants *variants, plaac_summary *summaries);

/* Effect columns of plaac_score_variant_effects: bit k (0..12) = the k-th double of plaac_summary in declaration order,
 * bit 13 = CORE change. */
#define PLAAC_EFFECT_LLR           (1 << 0)
#define PLAAC_EFFECT_CORE_SCORE    (1 << 1)
#define PLAAC_EFFECT_PRD_SCORE     (1 << 2)
#define PLAAC_EFFECT_HMM_ALL       (1 << 3)
#define PLAAC_EFFECT_HMM_VIT       (1 << 4)
#define PLAAC_EFFECT_FI_MEANHYDRO  (1 << 5)
#define PLAAC_EFFECT_FI_MEANCHARGE (1 << 6)
#define PLAAC_EFFECT_FI_MEANCOMBO  (1 << 7)
#define PLAAC_EFFECT_PAPA_COMBO    (1 << 8)
#define PLAAC_EFFECT_PAPA_PROP     (1 << 9)
#define PLAAC_EFFECT_PAPA_FI       (1 << 10)
#define PLAAC_EFFECT_PAPA_LLR      (1 << 11)
#define PLAAC_EFFECT_PAPA_LLR2     (1 << 12)
#define PLAAC_EFFECT_CORE_CHANGE   (1 << 13)

/* The effect of each variant against its wild type, in place of whole records (DESIGN.md section 11).  Arguments as
 * plaac_score_variants; columns is a non-zero mask of PLAAC_EFFECT_* bits.
 *   effects  HOST array (pinned or pageable) of nvar x popcount(columns) doubles, row-major: one row per variant in
 *            variant order, columns in ascending bit order.  Bits 0-12: variant.field - wild.field, one IEEE double
 *            subtraction and nothing else (NaN on either side gives NaN, -Inf - -Inf gives NaN, a PAPA centre that
 *            appears gives +Inf).  Bit 13: has_core(variant) - has_core(wild) as a double (+1 gained, -1 lost, 0
 *            unchanged), has_core meaning core_score is not NaN.
 *   wild     NULL, or nprot HOST records, each byte-identical to what plaac_score(codes, offsets, nprot) returns.
 * The variants' records and the wild-type records stay on the device; only the effects are copied back.  Errors, their
 * messages, the nvar == 0 case and the long-path rule are those of plaac_score_variants.  In addition PLAAC_E_INVALID
 * for columns == 0, a bit above 13, or a NULL effects with nvar > 0.  Reference bytes > 21 are scored as X: the effects
 * are written and the call then returns PLAAC_E_INVALID, as plaac_score does. */
int plaac_score_variant_effects(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                                const plaac_variants *variants, int32_t columns, double *effects, plaac_summary *wild);

/* ---- prion-like segments of the Viterbi parse (DESIGN.md section 12) ----------------------------------------------
 * A segment of protein i is a maximal run of residues whose Viterbi state is 1 (PrD-like): a maximal run of 1s of the
 * VIT column of per-residue mode.  start and end are 0-based, end inclusive (as prd_start / prd_end); score is
 * 0.0 + llr[aa[start]] + ... + llr[aa[end]] summed in residue order (the PRDscore rule, plaac.java:861-873), codes > 21
 * counting as X.  The segment that holds a protein's CORE therefore equals (prd_start, prd_end, prd_score) bit for bit,
 * and the longest segment's length is vit_maxrun. */
typedef struct plaac_segments {
    int64_t capacity;  /* in: entries start / end / score can hold */
    int64_t *first;    /* out: nprot + 1; the segments of protein i are [first[i], first[i+1]), complete even when
                          count > capacity */
    int32_t *start;    /* out: 0-based */
    int32_t *end;      /* out: 0-based, inclusive */
    double *score;     /* out: the PRDscore rule over the segment */
    int64_t count;     /* out: segments in the batch; the first min(count, capacity) are stored, in input order */
} plaac_segments;

/* Summary mode with the segment list of every protein.  codes / offsets / nprot as plaac_score; HOST buffers (pinned or
 * pageable) everywhere; blocks until done.  summaries: NULL (records are not copied back) or nprot records,
 * byte-identical to plaac_score's.  The segments are extracted on the device from the parse the summary kernels leave
 * behind and do not depend on the chunking, the long-path setting or the kernel variant.  Call again with
 * capacity = count when count > capacity.
 * PLAAC_E_INVALID for a negative capacity, a NULL first with nprot > 0, or a NULL start / end / score with
 * capacity > 0.  Reference bytes > 21 are scored as X: everything is written and the call then returns
 * PLAAC_E_INVALID, as plaac_score does.  nprot == 0: first[0] = 0, count = 0, PLAAC_OK. */
int plaac_score_segments(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                         plaac_summary *summaries, plaac_segments *segments);

/* ---- shuffled replicates: a composition-preserving null per protein (DESIGN.md section 13) -----------------------
 * Replicate r of reference protein i (length n) is rep[t] = ref[pi(t)], pi a bijection of [0, n) that is a pure function
 * of (seed, i, r, n): a 6-round cycle-walking Feistel network on [0, 2^b), 2^b the smallest power of two >= n, defined
 * in DESIGN.md section 13; the identity for n <= 1.  Bytes > 21 move like any other byte. */

/* Writes replicate `replicate` of `protein` (the protein's index in its batch, which selects the permutation) into
 * out[0 .. n): out[t] = codes[pi(t)], codes the protein's n residues.  Host only, no ctx or GPU needed.
 * PLAAC_E_INVALID for n < 0 or n >= 2^31, a negative protein or replicate, or NULL codes / out with n > 0. */
int plaac_shuffle_host(const uint8_t *codes, int64_t n, uint64_t seed, int64_t protein, int64_t replicate, uint8_t *out);

/* Column bit of plaac_null: replicates that have a CORE (the other bits are the PLAAC_EFFECT_* bits 0..12). */
#define PLAAC_NULL_HAS_CORE (1 << 13)

typedef struct plaac_null {
    int64_t replicates;      /* in: K >= 0 shuffles per selected protein */
    uint64_t seed;           /* in */
    int32_t columns;         /* in: non-zero mask of PLAAC_EFFECT_* bits 0..12, plus PLAAC_NULL_HAS_CORE */
    int32_t reserved;        /* in: must be 0 */
    int64_t nsel;            /* in: -1 = every protein of the batch, else the length of `proteins` */
    const int32_t *proteins; /* in: nsel reference indices (may repeat), or NULL when nsel == -1 */
    int64_t *counts;         /* out: nsel x popcount(columns), row-major, columns in ascending bit order */
    double *values;          /* out: NULL, or nsel x K x popcount(columns): the replicates' column values,
                                row j*K + r = replicate r of selected protein j */
} plaac_null;

/* Scores K shuffles of each selected protein, built on the device, and counts per protein and column the replicates that
 * reach the observed score.  codes / offsets / nprot: the reference batch, as plaac_score takes it.  For a double
 * column f a replicate counts when key(rep.f) >= key(obs.f), key(x) = isnan(x) ? -Inf : x (a missing CORE or PAPA ranks
 * lowest); PLAAC_NULL_HAS_CORE counts the replicates with a CORE (its value is 0 or 1).  The empirical p-value of a
 * column is (1 + count) / (1 + K).  observed: NULL or nsel records, observed[j] byte-identical to plaac_score's record
 * of protein proteins[j].  HOST buffers (pinned or pageable) everywhere; blocks until done.  Counts and values do not
 * depend on the chunking, the long-path setting, the kernel variant or the selection; chunks use the automatic long-path
 * threshold, as plaac_score_variants.
 * PLAAC_E_INVALID, with the offending index in plaac_last_error: replicates < 0, nsel < -1, reserved != 0, columns == 0
 * or a bit above 13, a selected index outside [0, nprot), NULL proteins with nsel >= 0, NULL counts with nsel != 0.
 * K == 0: counts are 0 and observed is written.  nprot == 0 or nsel == 0: PLAAC_OK, nothing written.  Reference bytes
 * > 21 are scored as X: everything is written and the call then returns PLAAC_E_INVALID, as plaac_score does. */
int plaac_score_shuffles(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                         plaac_null *null_spec, plaac_summary *observed);

/* Sequential shuffle null (Besag and Clifford, Biometrika 78:301, 1991; DESIGN.md section 14): as plaac_score_shuffles,
 * but each (selected protein, column) stops once h = stop_hits of its replicates have reached the observed score, after
 * at most K_max = null_spec->replicates replicates.  With hit(r) the counting rule of plaac_score_shuffles applied to
 * replicate r of the protein:
 *   L     = the smallest L in [1, K_max] with hit(0) + ... + hit(L-1) == h; K_max if there is none;
 *   count = hit(0) + ... + hit(L-1): h if the column stopped, below h otherwise.
 * Both are pure functions of (seed, reference index, columns, h, K_max): they do not depend on the selection's order or
 * repeats, the chunking, the long-path setting, the kernel variant or the round schedule.  With h > K_max nothing stops:
 * count equals plaac_score_shuffles' count for K = K_max, and L = K_max.  The p-value is h / L when count == h, and
 * (count + 1) / (K_max + 1) otherwise.  A protein is scored in rounds while any of its columns is below h, so a protein
 * with true p-value p costs about min(h / p, K_max) replicates.
 * null_spec: replicates = K_max; seed, columns, nsel, proteins as plaac_score_shuffles; reserved must be 0; counts
 * receives count (nsel x popcount(columns), row-major, columns in ascending bit order); values must be NULL.  scored
 * receives L in the same layout.  observed: NULL or nsel records, byte-identical to plaac_score's.  HOST buffers (pinned
 * or pageable); blocks until done.
 * PLAAC_E_INVALID as plaac_score_shuffles, and for stop_hits < 1, a non-NULL values, a NULL scored with nsel != 0.
 * K_max == 0: counts and scored are 0 and observed is written.  nsel == 0: PLAAC_OK, nothing written.  Reference bytes
 * > 21 are scored as X: everything is written and the call then returns PLAAC_E_INVALID. */
int plaac_score_shuffles_seq(plaac_ctx *ctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                             const plaac_null *null_spec, int64_t stop_hits, int64_t *scored, plaac_summary *observed);

/* ---- multi-GPU (SURVEY.md section 8e): proteins are independent, so the batch is cut into contiguous,
 * residue-balanced shards, one per ctx (each ctx on its own GPU), scored concurrently by one host thread per
 * ctx, each writing its records / per-residue rows straight into the caller's arrays at the input position.
 * No collective, no gather copy.  The reference has no counterpart (the jar is single-threaded). */

/* Shard plan: bounds[0..nshards], bounds[0] = 0, bounds[nshards] = nprot, shard k = proteins
 * [bounds[k], bounds[k+1]).  Balanced on (residues + 64 per protein).  Pure host arithmetic (no GPU needed). */
int plaac_shard_plan(const int64_t *offsets, int64_t nprot, int nshards, int64_t *bounds);

/* Same contract as plaac_score() with nctx contexts.  Returns the first non-zero shard return code
 * (its text is on that shard's ctx); all shards are always joined before returning. */
int plaac_score_multi(plaac_ctx *const *ctxs, int nctx, const uint8_t *codes, const int64_t *offsets, int64_t nprot,
                      plaac_summary *summaries, const plaac_residue_out *per_res);

/* The transport-lean form of plaac_score_multi (see plaac_score_packed): shards are cut on the lengths, a shard may
 * start in the middle of a word.  Compact output: every shard's candidate rows (its proteins with a CORE, or its top K)
 * are pulled onto the first context's GPU over NVLink / PCIe peer copies, ranked there as one set and copied to `hits`
 * once -- the only exchange between GPUs on the whole path. */
int plaac_score_multi_packed(plaac_ctx *const *ctxs, int nctx, const uint32_t *words, const int32_t *lengths, int64_t nprot,
                             int64_t nres, plaac_summary *summaries, const plaac_residue_out *per_res, plaac_hits *hits);

/* Shuffle nulls on nctx contexts (DESIGN.md section 15): the replicate axis is split, not the proteins.  Every ctx
 * scores every selected protein, ctx k the replicates [floor(K k / nctx), floor(K (k+1) / nctx)) of each (of each
 * round's span, for the sequential call, whose rounds run in lockstep on all ctxs).  counts, values, scored and
 * observed are byte-identical to plaac_score_shuffles / plaac_score_shuffles_seq on ctxs[0], for every nctx, whichever
 * devices the ctxs are on (several may share one) and whatever each ctx's chunk and long-path settings are; so are
 * they under each ctx's kernel variant, but for the PAPA columns (bits 8..12), whose bytes kernel variant 1 computes in
 * reference order (plaac_set_kernel_variant).  All ctxs must have been created with the same plaac_params.  nctx == 1
 * calls the single function.  Every ctx computes the observed records of the whole selection (only ctxs[0] writes them
 * to `observed`).
 * Errors: PLAAC_E_INVALID for nctx < 1, a NULL ctxs or a NULL ctxs[k] (text in plaac_last_error(NULL)), and as the
 * single call, before any device work, with this call's name and the text on ctxs[0].  Reference bytes > 21: everything
 * is written, then PLAAC_E_INVALID with the text on ctxs[0].  A CUDA error returns the first non-zero code in ctx order,
 * its text on that ctx.  Every host thread is joined before the call returns. */
int plaac_score_shuffles_multi(plaac_ctx *const *ctxs, int nctx, const uint8_t *codes, const int64_t *offsets,
                               int64_t nprot, plaac_null *null_spec, plaac_summary *observed);
int plaac_score_shuffles_seq_multi(plaac_ctx *const *ctxs, int nctx, const uint8_t *codes, const int64_t *offsets,
                                   int64_t nprot, const plaac_null *null_spec, int64_t stop_hits, int64_t *scored,
                                   plaac_summary *observed);

/* ---- GPU FASTA ingest and background counts (SURVEY.md section 8f, rows N2/N3) --------------------------------
 * Replaces fastareader (plaac.java:4302-4375) + string2aa (:1764-1769) + the terminal '*' strip (:758) for a whole
 * file image, and computeaafreq/isvalidprotein (:1655-1739) for the background counts.  Reader semantics are the
 * jar's: \n, \r, \r\n line ends; sequence lines are not trimmed; an empty line ends the record and everything up to
 * the next '>' line is skipped.  Records with an empty sequence are kept (offsets[i+1] == offsets[i]) so that names
 * stay aligned; the host prints no row for them (:762). */
typedef struct plaac_fasta_index {
    int64_t nrec;       /* records found in the text (may exceed max_rec: then only max_rec were stored) */
    int64_t nres;       /* residues written to codes */
} plaac_fasta_index;

/* HOST text in, HOST arrays out.  codes: capacity nbytes; offsets: max_rec+1; name_pos/name_len/flags: max_rec
 * (any of the three may be NULL).  flags bit 0: the jar trims this name (found after an empty line or at file start,
 * :4362); bit 1: a terminal '*' was stripped.  bg_counts (22 doubles, may be NULL) receives the residue counts of the
 * valid records exactly as computeaafreq(file) would (64-bit accumulation). */
int plaac_ingest_fasta(plaac_ctx *ctx, const char *text, int64_t nbytes, uint8_t *codes, int64_t *offsets,
                       int64_t *name_pos, int32_t *name_len, uint8_t *flags, int64_t max_rec, plaac_fasta_index *index,
                       double *bg_counts);

/* DEVICE text in, DEVICE arrays out (same capacities; d_bg_counts: 22 x uint64, may be NULL).  The outputs feed
 * plaac_score_device directly.  index is written on return (one small D2H).  d_flags must be 4-byte aligned and its
 * capacity a multiple of 4 bytes (bits are set with word-wide atomics). */
int plaac_ingest_fasta_device(plaac_ctx *ctx, const char *d_text, int64_t nbytes, uint8_t *d_codes, int64_t *d_offsets,
                              int64_t *d_name_pos, int32_t *d_name_len, uint8_t *d_flags, int64_t max_rec,
                              plaac_fasta_index *index, uint64_t *d_bg_counts);

/* FASTA text in, summary records out: plaac_ingest_fasta_device + plaac_score_device without the codes ever leaving
 * the GPU on the way in (H2D = the file bytes).  All pointers are HOST buffers: summaries, offsets, name_pos, name_len and flags as in
 * plaac_ingest_fasta (capacity max_rec), codes (capacity nbytes, may be NULL) receives the residue codes for the
 * string columns the host prints.  Replaces the whole loop of scoreallfastas (:755-948) for one file image. */
int plaac_score_fasta(plaac_ctx *ctx, const char *text, int64_t nbytes, int64_t max_rec, plaac_summary *summaries,
                      uint8_t *codes, int64_t *offsets, int64_t *name_pos, int32_t *name_len, uint8_t *flags,
                      plaac_fasta_index *index, double *bg_counts);

/* ---- on-device ranking and compact output (SURVEY.md section 8f, row N4) ---------------------------------------
 * The order the reference's web front end gives the table before it paginates (web/lib/server.rb:222-229):
 * COREscore descending, then LLR descending, rows without a CORE (COREscore NaN) last; equal rows keep input
 * order (the Ruby sort_by is unstable there, so any order of equal rows is one of its possible outputs).
 * order[k] = input index of the row ranked k; *n_core (may be NULL) = number of rows with a CORE, i.e. the head
 * order[0 .. n_core) is "every protein with a CORE, best first".  Values are compared at full precision (the web
 * compares the 3-decimal text).  A protein shorter than the core length has LLR = -Inf here and "NaN" in the printed
 * table (inf2nan, plaac.java:904/1008), which server.rb:225 sorts last within its COREscore group -- exactly where
 * -Inf sorts, so this IS the web order.  flags: reserved, must be 0. */
int plaac_rank_device(plaac_ctx *ctx, const plaac_summary *d_summaries, int64_t nprot, int flags, int32_t *d_order,
                      int64_t *n_core);
/* d_out[k] = d_summaries[d_order[k]] for k < count: ship the head of the ranking instead of 160 B x nprot.
 * Enqueued on the ctx stream (plaac_sync before reading). */
int plaac_gather_device(plaac_ctx *ctx, const plaac_summary *d_summaries, const int32_t *d_order, int64_t count,
                        plaac_summary *d_out);
/* HOST records in, HOST order out. */
int plaac_rank(plaac_ctx *ctx, const plaac_summary *summaries, int64_t nprot, int flags, int32_t *order, int64_t *n_core);

/* Host-side parameter chain for hosts that do not have their own (the C++ CLI, Python tests): what
 * plaac.java main computes between :310 and :518 -- bg/fg mixing with alpha (:449-458), the 1e-5
 * pseudo-frequency for X and * (:490-496), llr (:497-500), prionhmm1/prionhmm0 (:968-1001) through
 * hmm.initialize (:2893-2935), loglut and lodpapa1 (:279-299), aahydro2 (:90).  Uses the C library's
 * log/exp.  bg_counts: the 22 numbers of `bgf` (:374-384) or NULL (all zero); fg_freq: 22 numbers or
 * NULL for the built-in prd_freq_scer_28 (:269).  alpha outside [0,1] becomes 1 (:444-447).
 * info (optional, 4 x 22 doubles): fg_used, bg_scer, bg_input, bg_used as printed at :506-509. */
int plaac_params_init(plaac_params *out, double alpha, const double *bg_counts, const double *fg_freq,
                      int core_len, int ww1, int ww2, int ww3, int adjust_prolines, double *info);

/* residue encoding on the host side of the ABI (aatoint/string2aa, :1508-1534,
 * :1764-1769): n chars -> n codes; does NOT strip the stop codon. */
void plaac_encode_host(const char *chars, int64_t n, uint8_t *codes);

/* Tuning/testing knob for plaac_score(): upper bounds of one device chunk (0 = keep default). */
int plaac_set_chunk(plaac_ctx *ctx, int64_t max_residues, int64_t max_proteins);

/* Long-sequence path (BASELINE config 5).  Summary mode: the record of a protein of at least min_len residues is
 * computed chunk-parallel.  Its HMM columns (forward score, Viterbi parse and score) come from the thread-block cluster
 * of the per-residue mode below, in records-only form (csrc/long_residue.cuh).  Beside it, two CTAs per protein cut it
 * into <= 384 chunks (csrc/long_kernel.cuh): one computes the plain fp64 sums and the MW and LLR searches, the other the
 * window columns.  Every chunk of a recurrence or sum is re-run in the jar's own binade, where every rounding commutes
 * with the chunk's shift, so the combined values have the jar's bits.  Two small kernels then compute longestrun, the
 * CORE search and the two HMM scores.  The path is a latency device (whole CTAs per protein are less efficient per
 * residue than the bucketed kernel).  min_len > 0: fixed threshold (default 8192, where a lane's sequential walk of
 * the protein, ~1.4 ms, exceeds what a whole typical batch takes; raised to 1024 / four times the longest window if
 * smaller).  min_len = -1: automatic threshold per batch -- the smallest length, at least 1024 residues and at least
 * ntotal/81600 + 220 (the walk must be a visible part of the batch's time), that leaves no more long proteins than the
 * GPU has SMs; best latency for small proteomes (a yeast-sized set: 0.9 instead of 1.4 ms) at the price of one more
 * host synchronisation per device-resident call.  min_len = 0: path off.  warm: warm-up length in residues of the
 * cluster kernel's forward (and backward) chunks, rounded up to whole chunks; 0 keeps the current value (default 256),
 * a negative value is taken by its magnitude.  A short warm-up only costs time: -1 gives the shortest, with which
 * nearly every chunk is redone sequentially (testing).  Both paths give the same bytes in every column (the
 * recurrences by the binade-frame argument, the window columns because their sums are exact on a 2^-41 grid), so
 * records do not depend on the setting, the batching or the sharding.
 * Per-residue mode (plotsomefastas :610-647 on long proteins): the same threshold sends a protein to one thread-block
 * cluster (csrc/long_residue.cuh: 1 CTA below 32768 residues, 8 above; forward, backward and Viterbi recurrences
 * chunk-parallel in the jar's binade with an exact carry over the chunk boundaries, relayed between the CTAs through
 * distributed shared memory), and the per-residue arrays are byte for byte those of the single-lane walk; the automatic
 * threshold then admits half as many proteins (two CTAs per long protein run side by side). */
int plaac_set_long_path(plaac_ctx *ctx, int64_t min_len, int warm);

/* Kernel selection for testing: 0 = automatic (default), 1 = the reference-order anchor kernel (one fused
 * kernel, every recurrence in plaac.java's operation order, slower), 2 / 3 = the throughput kernels (role-split;
 * 3 is 2 with fewer issue slots per residue and is what 0 selects; both need loglut[0] == ln2 and le0 == le[0],
 * true for tables built as plaac.java builds them). */
int plaac_set_kernel_variant(plaac_ctx *ctx, int variant);

/* Accounting for benchmarks: kernels launched by this ctx so far, and the
 * CUDA-event time (ms) the scoring kernel(s) of the LAST plaac_score_device
 * call took on the ctx stream (valid after plaac_sync). */
typedef struct plaac_stats {
    int64_t kernel_launches;   /* all kernels of this library launched by the ctx */
    int64_t score_launches;    /* launches of the dominant scoring kernel */
    float last_total_ms;       /* whole pipeline of the last device call */
    float last_score_ms;       /* dominant kernel of the last device call */
    int64_t last_padded_slots; /* 16-byte lane slots in the bucketed stream of the last call */
    int64_t long_proteins;     /* proteins scored by the long-sequence path so far */
    int64_t long_redone_chunks; /* chunks of that path's cluster kernel redone sequentially although they had frames
                                   (their warm-up had not coalesced) */
} plaac_stats;
int plaac_get_stats(plaac_ctx *ctx, plaac_stats *out);

#ifdef __cplusplus
}
#endif
#endif
