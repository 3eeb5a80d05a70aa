// Prion-like segments of the Viterbi parse (plaac_score_segments, DESIGN.md section 12): every maximal run of
// PrD-state residues of every protein, read from the parse the summary kernels leave in the slot.
//   bucketed proteins: BatchView::tbw, the Viterbi bits of residue i of rank r = 32 b + lane in bit (i & 15) of word
//                      (chunk_base[b] + (i >> 4)) * 32 + lane -- the layout of every summary kernel (v1, v2, v3)
//   long-path proteins: the 32-bit words k_long_final writes at vit + (scratch_off >> 5), bit (i & 31) of word i >> 5
// Per chunk, on the slot's stream, after the CORE search and after the long-path streams have joined:
//   k_seg_count + k_seg_count_long -> launch_scan (first) -> k_seg_bounds + k_seg_bounds_long -> k_seg_score
// Entries at or above the capacity are not stored; first[np] always holds the chunk's true total.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace plaac {

constexpr int kSegLongThreads = 256;

struct SegArgs {
    BatchView bv;                    // bucketed parse, order, chunk_base, offsets (chunk-relative), long_min
    const uint8_t* codes;            // the chunk's residue codes, protein p at offsets[p] - bv.off_base
    const DeviceTables* tabs;
    const int32_t* long_list;        // long-path proteins of the chunk (k_long_select), or NULL
    const int64_t* long_off;         // their scratch offsets
    const uint32_t* long_vit;        // their parse words
    int64_t nlong;
    int32_t* count;                  // np: segments per protein
    const int64_t* first;            // np + 1: exclusive scan of count
    int32_t* prot;                   // cap entries each
    int32_t* start;
    int32_t* end;
    double* score;
    int64_t cap;
};

// Walks the runs of one protein's parse whose start lies in words [j_lo, j_hi) (W = 16 or 32 bits per word, at stride
// `stride`) and calls f(start, end) for each, in order; a run is followed past j_hi to its end.  entering: the word before
// j_lo ends in a 1, so the run that continues into j_lo started before it and is not this walk's.  A run start is
// bits & ~((bits << 1) | carry); a run ending at a word's top bit continues if the next word's bit 0 is set.
template <int W, typename F>
__device__ __forceinline__ void seg_walk(const uint32_t* __restrict__ vw, size_t stride, int n, int j_lo, int j_hi, bool entering,
                                         F f)
{
    constexpr uint32_t kFull = (W == 32) ? 0xffffffffu : ((1u << W) - 1u);
    const int jlast = (n - 1) / W;
    auto word = [&](int j) -> uint32_t {
        const uint32_t v = vw[(size_t)j * stride] & kFull;
        return j == jlast ? v & ((2u << ((n - 1) % W)) - 1u) : v;
    };
    if (n <= 0 || j_lo >= j_hi || j_lo > jlast) return;
    int open = entering ? -2 : -1;  // -2: the entering run (not reported), -1: none
    uint32_t cur = word(j_lo), cin = entering ? 1u : 0u;
    for (int j = j_lo; j < j_hi; j++) {
        const uint32_t nxt = (j + 1 <= jlast) ? word(j + 1) : 0u;
        uint32_t s = cur & ~((cur << 1) | cin);
        uint32_t e = cur & ~(cur >> 1);
        const int base = j * W;
        while (e) {
            const int p = __ffs((int)e) - 1;
            e &= e - 1;
            if (open == -1) {
                open = base + __ffs((int)s) - 1;
                s &= s - 1;
            }
            if (p == W - 1 && (nxt & 1u)) break;  // continues into the next word (always the word's last end)
            if (open >= 0) f(open, base + p);
            open = -1;
        }
        cin = cur >> (W - 1);
        cur = nxt;
    }
    if (open < 0) return;
    for (int j = j_hi; j <= jlast; j++) {  // word j's bit 0 is set
        const uint32_t zeros = ~word(j) & kFull;
        if (zeros) {
            f(open, j * W + __ffs((int)zeros) - 2);
            return;
        }
    }
    f(open, n - 1);
}

__device__ __forceinline__ int seg_count_words(uint32_t bits, uint32_t carry) { return __popc(bits & ~((bits << 1) | carry)); }

// Segments per bucketed protein: one thread per rank (the lanes of a warp read the lane-strided words of one bucket).
__global__ void __launch_bounds__(256) k_seg_count(SegArgs g)
{
    const int64_t rank = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (rank >= g.bv.nprot) return;
    const int32_t prot = g.bv.order[rank];
    const int64_t len = g.bv.offsets[prot + 1] - g.bv.offsets[prot];
    const int n = (int)eff_len(len, g.bv.long_min);
    if (n == 0 && len != 0) return;  // k_seg_count_long
    const int64_t b = rank >> 5;
    const uint32_t* vw = g.bv.tbw + g.bv.chunk_base[b] * 32 + (rank & 31);
    int cnt = 0;
    uint32_t carry = 0;
    const int jlast = (n - 1) >> 4;
    for (int j = 0; j <= jlast && n > 0; j++) {
        uint32_t bits = vw[(size_t)j * 32] & 0xffffu;
        if (j == jlast) bits &= (2u << ((n - 1) & 15)) - 1u;
        cnt += seg_count_words(bits, carry);
        carry = (bits >> 15) & 1u;
    }
    g.count[prot] = cnt;
}

// Per-thread contiguous ranges of a long protein's 32-bit words; the range's run starts, carry from the word before it.
__device__ __forceinline__ int seg_long_range_count(const uint32_t* vw, int n, int w_lo, int w_hi)
{
    const int jlast = (n - 1) >> 5;
    uint32_t carry = w_lo > 0 ? vw[w_lo - 1] >> 31 : 0u;
    int cnt = 0;
    for (int j = w_lo; j < w_hi; j++) {
        uint32_t bits = vw[j];
        if (j == jlast) bits &= (2u << ((n - 1) & 31)) - 1u;
        cnt += seg_count_words(bits, carry);
        carry = bits >> 31;
    }
    return cnt;
}

// Block-level exclusive scan of one int per thread (kSegLongThreads); returns the thread's base, *total the sum.
__device__ __forceinline__ int seg_block_scan(int v, int* total)
{
    __shared__ int warp_sum[kSegLongThreads / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) warp_sum[wid] = inc;
    __syncthreads();
    int base = 0, all = 0;
#pragma unroll
    for (int k = 0; k < kSegLongThreads / 32; k++) {
        base += (k < wid) ? warp_sum[k] : 0;
        all += warp_sum[k];
    }
    *total = all;
    return base + inc - v;
}

// Segments per long-path protein: one block per protein, the threads' counts combined in the block.
__global__ void __launch_bounds__(kSegLongThreads) k_seg_count_long(SegArgs g)
{
    const int32_t prot = g.long_list[blockIdx.x];
    const int n = (int)(g.bv.offsets[prot + 1] - g.bv.offsets[prot]);
    const uint32_t* vw = g.long_vit + (g.long_off[blockIdx.x] >> 5);
    const int nwords = (n + 31) >> 5;
    const int per = (nwords + kSegLongThreads - 1) / kSegLongThreads;
    const int w_lo = min(nwords, (int)threadIdx.x * per), w_hi = min(nwords, w_lo + per);
    int total;
    seg_block_scan(seg_long_range_count(vw, n, w_lo, w_hi), &total);
    if (threadIdx.x == 0) g.count[prot] = total;
}

__device__ __forceinline__ void seg_put(const SegArgs& g, int64_t idx, int32_t prot, int s, int e)
{
    if (idx >= g.cap) return;
    g.prot[idx] = prot;
    g.start[idx] = s;
    g.end[idx] = e;
}

// Bounds of the bucketed proteins' segments: one thread per rank.
__global__ void __launch_bounds__(256) k_seg_bounds(SegArgs g)
{
    const int64_t rank = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (rank >= g.bv.nprot) return;
    const int32_t prot = g.bv.order[rank];
    const int64_t len = g.bv.offsets[prot + 1] - g.bv.offsets[prot];
    const int n = (int)eff_len(len, g.bv.long_min);
    if (n == 0) return;
    int64_t idx = g.first[prot];
    if (idx >= g.cap) return;
    const uint32_t* vw = g.bv.tbw + g.bv.chunk_base[rank >> 5] * 32 + (rank & 31);
    seg_walk<16>(vw, 32, n, 0, ((n - 1) >> 4) + 1, false, [&](int s, int e) { seg_put(g, idx++, prot, s, e); });
}

// Bounds of the long-path proteins' segments: one block per protein; a thread writes the runs that start in its range.
__global__ void __launch_bounds__(kSegLongThreads) k_seg_bounds_long(SegArgs g)
{
    const int32_t prot = g.long_list[blockIdx.x];
    const int n = (int)(g.bv.offsets[prot + 1] - g.bv.offsets[prot]);
    const uint32_t* vw = g.long_vit + (g.long_off[blockIdx.x] >> 5);
    const int nwords = (n + 31) >> 5;
    const int per = (nwords + kSegLongThreads - 1) / kSegLongThreads;
    const int w_lo = min(nwords, (int)threadIdx.x * per), w_hi = min(nwords, w_lo + per);
    int total;
    const int mine = seg_long_range_count(vw, n, w_lo, w_hi);
    int64_t idx = g.first[prot] + seg_block_scan(mine, &total);
    if (mine == 0 || idx >= g.cap) return;
    const bool entering = w_lo > 0 && (vw[w_lo - 1] >> 31);  // (word w_lo - 1 is never the last word)
    seg_walk<32>(vw, 1, n, w_lo, w_hi, entering, [&](int s, int e) { seg_put(g, idx++, prot, s, e); });
}

// Scores: one thread per stored segment, 0.0 + llr[aa[start]] + ... + llr[aa[end]] in residue order (a dependent DADD
// chain, as PRDscore, plaac.java:861-873).
__global__ void __launch_bounds__(128) k_seg_score(SegArgs g, int64_t np)
{
    __shared__ double llr_s[32];
    if (threadIdx.x < 32) llr_s[threadIdx.x] = g.tabs->llr[threadIdx.x];
    __syncthreads();
    const int64_t stored = min(g.first[np], g.cap);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < stored; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t prot = g.prot[i];
        const uint8_t* __restrict__ src = g.codes + (g.bv.offsets[prot] - g.bv.off_base);
        const int e = g.end[i];
        double sc = 0.0;
        for (int k = g.start[i]; k <= e; k++) {
            const uint32_t cd = src[k];
            sc = sc + llr_s[cd > 21u ? 0u : cd];
        }
        g.score[i] = sc;
    }
}

}  // namespace plaac
