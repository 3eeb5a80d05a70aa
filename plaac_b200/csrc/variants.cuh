// Sequence variants built on the device (plaac_score_variants): the reference batch is uploaded once per call, and each
// chunk of the variant list is expanded from it into the slot's code buffer that k_pack reads, so only the substitution
// list crosses the host link.  Per chunk, on the slot's stream:
//   k_variant_lengths -> launch_scan (offsets) -> k_variant_expand -> k_variant_apply -> run_batch
//   [-> k_variant_effect for plaac_score_variant_effects].
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lean.cuh"  // rec_has_core

namespace plaac {

constexpr int kExpandThreads = 256;
constexpr int kExpandSteps = 16;                                 // 16-byte stores per thread
constexpr int kExpandTile = kExpandThreads * 16 * kExpandSteps;  // output bytes per block

// len[v] = length of variant v's reference protein.
__global__ void __launch_bounds__(256)
k_variant_lengths(const int32_t* __restrict__ protein, int64_t nvar, const int64_t* __restrict__ ref_off,
                  int32_t* __restrict__ len)
{
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvar) return;
    const int32_t p = protein[v];
    len[v] = (int32_t)(ref_off[p + 1] - ref_off[p]);
}

// Last index v in [lo, hi] with a[v] <= x (a non-decreasing, a[lo] <= x).
template <typename T>
__device__ __forceinline__ int64_t last_not_above(const T* __restrict__ a, int64_t lo, int64_t hi, int64_t x)
{
    while (lo < hi) {
        const int64_t mid = lo + (hi - lo + 1) / 2;
        if ((int64_t)a[mid] <= x)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// Writes codes[x0 .. x0 + 16) (an aligned 16-byte block, clipped at nres); v is the variant that owns x0.  Inside one
// variant the bytes come from five aligned 4-byte loads of the reference (L1/L2-resident: a saturation scan reads one
// protein 19 n times); a block across a variant boundary or the end of the chunk goes byte by byte.
__device__ __forceinline__ void expand16(const uint8_t* __restrict__ ref, const int64_t* __restrict__ ref_off,
                                         int64_t ref_base, const int32_t* __restrict__ protein,
                                         const int64_t* __restrict__ off, int64_t v, int64_t x0, int64_t nres,
                                         uint8_t* __restrict__ codes)
{
    int64_t vb = off[v], ve = off[v + 1];
    const uint8_t* src = ref + (ref_off[protein[v]] - ref_base);
    uint32_t w[4] = {0, 0, 0, 0};
    if (x0 + 16 <= ve) {
        const uint8_t* s = src + (x0 - vb);
        const uint32_t* a = (const uint32_t*)((uintptr_t)s & ~(uintptr_t)3);
        const uint32_t sh = 8u * (uint32_t)((uintptr_t)s & 3);
        uint32_t r[5];
#pragma unroll
        for (int i = 0; i < 5; i++) r[i] = __ldg(a + i);
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = __funnelshift_r(r[i], r[i + 1], sh);
        *(uint4*)(codes + x0) = make_uint4(w[0], w[1], w[2], w[3]);
        return;
    }
    const int n = (int)min((int64_t)16, nres - x0);
    for (int k = 0; k < n; k++) {
        const int64_t x = x0 + k;
        while (x >= ve) {  // (skips empty variants)
            v++;
            vb = ve;
            ve = off[v + 1];
            src = ref + (ref_off[protein[v]] - ref_base);
        }
        w[k >> 2] |= (uint32_t)src[x - vb] << (8 * (k & 3));
    }
    if (n == 16)
        *(uint4*)(codes + x0) = make_uint4(w[0], w[1], w[2], w[3]);
    else
        for (int k = 0; k < n; k++) codes[x0 + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
}

// codes[off[v] .. off[v+1]) = reference residues of protein[v], for the nres residues of the chunk.  One block per
// 64 KB output tile whatever the lengths: the block finds the variants its tile spans by binary search in the offsets
// (a chain of dependent L2 loads, paid once per tile), then each thread writes 16 aligned 16-byte blocks, 4 KB apart,
// searching only between its previous variant and the tile's last.  Bytes behind nres are left as they are (the slack
// k_pack reads stays defined).
__global__ void __launch_bounds__(kExpandThreads)
k_variant_expand(const uint8_t* __restrict__ ref, const int64_t* __restrict__ ref_off, int64_t ref_base,
                 const int32_t* __restrict__ protein, const int64_t* __restrict__ off, int64_t nvar, int64_t nres,
                 uint8_t* __restrict__ codes)
{
    __shared__ int64_t s_range[2];
    const int64_t t0 = (int64_t)blockIdx.x * kExpandTile;
    if (threadIdx.x < 2) {
        const int64_t x = threadIdx.x == 0 ? t0 : min(t0 + kExpandTile, nres) - 1;
        s_range[threadIdx.x] = last_not_above(off, 0, nvar - 1, x);
    }
    __syncthreads();
    int64_t v = s_range[0];
    for (int step = 0; step < kExpandSteps; step++) {
        const int64_t x0 = t0 + (int64_t)step * (kExpandThreads * 16) + 16 * (int64_t)threadIdx.x;
        if (x0 >= nres) return;
        v = last_not_above(off, v, s_range[1], x0);
        expand16(ref, ref_off, ref_base, protein, off, v, x0, nres, codes);
    }
}

// One thread per substitution j of the chunk: codes[off[v] + pos[j]] = code[j], v the variant that owns j (first_sub
// is the chunk's slice of the caller's array, fs0 its first entry).  Runs after k_variant_expand in stream order.
__global__ void __launch_bounds__(256)
k_variant_apply(const int64_t* __restrict__ first_sub, int64_t fs0, int64_t nvar, const int32_t* __restrict__ pos,
                const uint8_t* __restrict__ code, int64_t nsub, const int64_t* __restrict__ off, uint8_t* __restrict__ codes)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nsub) return;
    const int64_t v = last_not_above(first_sub, 0, nvar - 1, fs0 + j);
    codes[off[v] + pos[j]] = code[j];
}

// plaac_score_variant_effects: out[v * k + c] = effect of variant v in the c-th set bit of `columns` (k of them), against
// the wild-type record of its reference protein (wild[protein[v]]).  One thread per output element, so the row-major
// stores coalesce; the record reads are 160-byte-strided gathers.  Bits 0..12 index the doubles of plaac_summary from
// llr on; bit 13 is the CORE change.  Runs after run_batch in stream order.
constexpr int kEffectCoreChange = 13;

__global__ void __launch_bounds__(256)
k_variant_effect(const plaac_summary* __restrict__ rec, const plaac_summary* __restrict__ wild,
                 const int32_t* __restrict__ protein, int64_t nvar, uint32_t columns, double* __restrict__ out)
{
    const int k = __popc(columns);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nvar * k) return;
    const int64_t v = e / k;
    const int f = (int)__fns(columns, 0, (int)(e - v * k) + 1);  // position of the (c+1)-th set bit
    const plaac_summary& a = rec[v];
    const plaac_summary& b = wild[protein[v]];
    out[e] = f == kEffectCoreChange ? (double)rec_has_core(a) - (double)rec_has_core(b) : __dsub_rn((&a.llr)[f], (&b.llr)[f]);
}

}  // namespace plaac
