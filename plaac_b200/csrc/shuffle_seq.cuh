// Sequential shuffle nulls (plaac_score_shuffles_seq, DESIGN.md section 14): replicates are scored in rounds
// [r0, r1) over a list of the selected proteins that are still active, and a (protein, column) stops at the replicate
// that brings its hits to h.  Per chunk of a round, on the slot's stream, the shuffle input form of shuffle.cuh runs with
// k_shuffle_flags in place of k_shuffle_tally; once per round (slice of the list), on one stream:
//   k_shuffle_stop -> launch_scan (active flags) -> k_shuffle_compact.
// On several ctxs (plaac_score_shuffles_seq_multi, DESIGN.md section 15) each ctx flags its part of the round's span, and
// k_shuffle_stop runs twice per slice: with h above any count, to count each row's hits in the part, then from the host's
// base counts, to find the replicate of the h-th hit in the part where a row reaches it.  The list stays on the host.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "shuffle.cuh"

namespace plaac {

// One thread per (replicate t, column c) of the chunk, as k_shuffle_tally.  The chunk is [q0, q0 + np) of the round's
// flattened index q = a * W + (r - r0), a the replicate's entry in the round's list (act[a] = its selection index, which
// indexes the observed records obs).  A hit sets bit r - r0 of row a * k + c of the round's flags (wpr words per row).
// The lanes of a warp that share a word OR their bits together first, and one atomicOr per word adds them, so the flags
// do not depend on the order of the chunks or slots.  Runs after run_batch.
__global__ void __launch_bounds__(256)
k_shuffle_flags(const plaac_summary* __restrict__ rec, const plaac_summary* __restrict__ obs, const int32_t* __restrict__ act,
                int64_t q0, int64_t W, int64_t np, uint32_t columns, int64_t wpr, uint32_t* __restrict__ flags)
{
    const int k = __popc(columns);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t word = -1;
    uint32_t bit = 0;
    if (e < np * k) {
        const int64_t t = e / k;
        const int c = (int)(e - t * k);
        const int f = (int)__fns(columns, 0, c + 1);  // position of the (c+1)-th set bit
        const int64_t q = q0 + t, a = q / W, r = q - a * W;
        const plaac_summary& x = rec[t];
        bool hit;
        if (f == kNullHasCore) {
            hit = rec_has_core(x);
        } else {
            const double v = (&x.llr)[f], o = (&obs[act[a]].llr)[f];
            hit = (v != v ? -INFINITY : v) >= (o != o ? -INFINITY : o);
        }
        word = (a * k + c) * wpr + (r >> 5);
        bit = hit ? 1u << (r & 31) : 0u;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, word);
    if (__ballot_sync(0xffffffffu, bit != 0) & peers) {  // (the same for every lane of the group)
        const uint32_t bits = __reduce_or_sync(peers, bit);
        if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicOr(flags + word, bits);
    }
}

// One warp per (entry a of the list, column c), for the round's replicates [r0, r1): the row's hits are counted word by
// word (__popc and a warp prefix sum).  A row that has not stopped and reaches h stops at the replicate of its
// (h - count)-th hit: scored = r0 + that bit's position + 1, count = h.  Otherwise count += hits and scored = r1, and
// the entry stays active (live[a] = 1) unless r1 is the last replicate kmax.  count and scored are indexed by the
// selection index act[a] * k + c.
__global__ void __launch_bounds__(256)
k_shuffle_stop(const uint32_t* __restrict__ flags, const int32_t* __restrict__ act, int64_t nact, int k, int64_t wpr,
               int64_t h, int64_t r0, int64_t r1, int64_t kmax, int64_t* __restrict__ count, int64_t* __restrict__ scored,
               int32_t* __restrict__ live)
{
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // row a * k + c
    const int lane = threadIdx.x & 31;
    if (w >= nact * k) return;
    const int64_t a = w / k, slot = (int64_t)act[a] * k + (w - a * k);
    int64_t n = count[slot];
    if (n >= h) return;  // stopped in an earlier round
    const uint32_t* row = flags + w * wpr;
    for (int64_t w0 = 0; w0 < wpr; w0 += 32) {
        const uint32_t x = w0 + lane < wpr ? row[w0 + lane] : 0u;
        const int p = __popc(x);
        int incl = p;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        const int tot = __shfl_sync(0xffffffffu, incl, 31);
        if (n + tot >= h) {
            const int need = (int)(h - n);  // 1 .. tot
            if (lane == __ffs(__ballot_sync(0xffffffffu, incl >= need)) - 1) {
                count[slot] = h;
                scored[slot] = r0 + (w0 + lane) * 32 + (int64_t)__fns(x, 0, need - (incl - p)) + 1;
            }
            return;
        }
        n += tot;
    }
    if (lane == 0) {
        count[slot] = n;
        scored[slot] = r1;
        if (r1 < kmax) live[a] = 1;
    }
}

// The next round's list: out[0] = the number of active entries, out[1 + pos[a]] = act[a] for the active ones (pos the
// exclusive scan of live), in list order.
__global__ void __launch_bounds__(256)
k_shuffle_compact(const int32_t* __restrict__ live, const int64_t* __restrict__ pos, const int32_t* __restrict__ act, int64_t n,
                  int32_t* __restrict__ out)
{
    const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a == 0) out[0] = (int32_t)pos[n];
    if (a < n && live[a]) out[1 + pos[a]] = act[a];
}

}  // namespace plaac
