// Shuffled replicates built on the device (plaac_score_shuffles, DESIGN.md section 13): the reference batch is uploaded
// once per call (variants_prepare), and each chunk -- a range [q0, q0 + np) of the flattened replicate index
// q = j * K + r (replicate r of selected protein j) -- is expanded from it into the slot's code buffer that k_pack reads.
// Per chunk, on the slot's stream:
//   k_shuffle_prep -> launch_scan (offsets) -> k_shuffle_expand -> run_batch -> k_shuffle_tally.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lean.cuh"  // rec_has_core
#include "shuffle.h"
#include "variants.cuh"  // last_not_above, kExpand*

namespace plaac {

// What k_shuffle_expand needs of one replicate: where its protein starts in the uploaded reference, and its permutation.
struct ShuffleRep {
    int64_t src;
    ShuffleKey key;
};

// One thread per replicate t of the chunk: its reference protein i (sel: the chunk's slice sel[j0 ..] of the selection,
// NULL for every protein of the batch), length and permutation.  q = j * K + (r - r0): a round of
// plaac_score_shuffles_seq scores replicates [r0, r0 + K); plaac_score_shuffles passes r0 = 0.
__global__ void __launch_bounds__(256)
k_shuffle_prep(const int32_t* __restrict__ sel, int64_t j0, int64_t q0, int64_t K, int64_t r0, int64_t np,
               const int64_t* __restrict__ ref_off, uint64_t seed, int32_t* __restrict__ len, ShuffleRep* __restrict__ rep)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= np) return;
    const int64_t q = q0 + t, j = q / K, r = r0 + q - j * K;
    const int64_t i = sel ? (int64_t)sel[j - j0] : j;
    const int64_t b = ref_off[i], n = ref_off[i + 1] - b;
    len[t] = (int32_t)n;
    ShuffleRep o;
    o.src = b - ref_off[0];
    o.key = shuffle_key(seed, i, r, n);
    rep[t] = o;
}

// codes[off[t] + x] = ref[src_t + pi_t(x)] for the nres residues of the chunk, tiled as k_variant_expand: one block per
// 64 KB output tile, each thread 16 aligned 16-byte blocks 4 KB apart.  Each byte is a gather from the L1/L2-resident
// reference.  Bytes behind nres are left as they are (the slack k_pack reads stays defined).
__global__ void __launch_bounds__(kExpandThreads)
k_shuffle_expand(const uint8_t* __restrict__ ref, const ShuffleRep* __restrict__ rep, const int64_t* __restrict__ off,
                 int64_t np, int64_t nres, uint8_t* __restrict__ codes)
{
    __shared__ int64_t s_range[2];
    const int64_t t0 = (int64_t)blockIdx.x * kExpandTile;
    if (threadIdx.x < 2) {
        const int64_t x = threadIdx.x == 0 ? t0 : min(t0 + kExpandTile, nres) - 1;
        s_range[threadIdx.x] = last_not_above(off, 0, np - 1, x);
    }
    __syncthreads();
    int64_t v = s_range[0];
    for (int step = 0; step < kExpandSteps; step++) {
        const int64_t x0 = t0 + (int64_t)step * (kExpandThreads * 16) + 16 * (int64_t)threadIdx.x;
        if (x0 >= nres) return;
        v = last_not_above(off, v, s_range[1], x0);
        const int n = (int)min((int64_t)16, nres - x0);
        uint64_t lo = 0, hi = 0;  // (two words, not an array: a run-time index would put it on the stack)
        int64_t vb = off[v], ve = off[v + 1];
        ShuffleRep p = rep[v];
        for (int k = 0; k < n; k++) {
            const int64_t x = x0 + k;
            while (x >= ve) {  // (skips empty replicates)
                v++;
                vb = ve;
                ve = off[v + 1];
                p = rep[v];
            }
            const uint64_t c = __ldg(ref + p.src + shuffle_index(p.key, (uint32_t)(x - vb)));
            if (k < 8)
                lo |= c << (8 * k);
            else
                hi |= c << (8 * (k - 8));
        }
        if (n == 16)
            *(uint4*)(codes + x0) = make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
        else
            for (int k = 0; k < n; k++) codes[x0 + k] = (uint8_t)((k < 8 ? lo : hi) >> (8 * (k & 7)));
    }
}

constexpr int kNullHasCore = 13;

// One thread per (replicate t, column c) of the chunk, c the c-th set bit f of `columns` (k of them): the replicate counts
// when key(rep.f) >= key(obs.f), key(x) = isnan(x) ? -Inf : x, obs = the observed record of its selected protein j;
// f == 13 counts replicates with a CORE.  counts[j * k + c] gathers the chunk's hits with integer atomics (exact, so the
// result does not depend on their order), summed first over the lanes of a warp that share the counter.  values, when
// not NULL, receives the chunk's rows: values[t * k + c] = rep.f (0 or 1 for f == 13).  Runs after run_batch.
__global__ void __launch_bounds__(256)
k_shuffle_tally(const plaac_summary* __restrict__ rec, const plaac_summary* __restrict__ obs, int64_t q0, int64_t K,
                int64_t np, uint32_t columns, unsigned long long* __restrict__ counts, double* __restrict__ values)
{
    const int k = __popc(columns);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = e < np * k;
    int64_t slot = -1;
    bool hit = false;
    if (live) {
        const int64_t t = e / k;
        const int c = (int)(e - t * k);
        const int f = (int)__fns(columns, 0, c + 1);  // position of the (c+1)-th set bit
        const int64_t j = (q0 + t) / K;
        const plaac_summary& a = rec[t];
        double v;
        if (f == kNullHasCore) {
            hit = rec_has_core(a);
            v = hit ? 1.0 : 0.0;
        } else {
            v = (&a.llr)[f];
            const double o = (&obs[j].llr)[f];
            hit = (v != v ? -INFINITY : v) >= (o != o ? -INFINITY : o);
        }
        if (values) values[e] = v;
        slot = j * k + c;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, slot);
    const unsigned hits = __ballot_sync(0xffffffffu, hit) & peers;
    if (live && hits && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(counts + slot, (unsigned long long)__popc(hits));
}

}  // namespace plaac
