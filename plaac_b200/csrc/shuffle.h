// The composition-preserving shuffle of plaac_score_shuffles and plaac_shuffle_host (DESIGN.md section 13), compiled by
// the device kernels and the host alike so that a replicate is the same sequence wherever it is built.
//
// Replicate r of reference protein i (length n) is rep[t] = ref[pi(t)], t in [0, n), where pi is a bijection of [0, n)
// and a pure function of (seed, i, r, n):
//   n <= 1: the identity.
//   b = bit length of n - 1 (so 2^(b-1) < n <= 2^b), the Feistel domain is [0, 2^b).
//   s = mix64(seed + G) ^ i;  s = mix64(s + G) ^ r;  key[k] = low 32 bits of mix64(s + (k + 1) G), k = 0..5
//     (G = 0x9E3779B97F4A7C15, mix64 = the splitmix64 finaliser).
//   Round k (k = 0..5) on x in [0, 2^b): w = b/2 (k even) or b - b/2 (k odd), R = low w bits, L = the other b - w;
//     x = (R << (b - w)) | (L ^ (mix32(R ^ key[k]) & (2^(b - w) - 1)))   (mix32 = the lowbias32 finaliser).
//   pi(t) = the Feistel network applied to t, again and again until the value is below n (cycle walking).
// Only 32/64-bit integer operations, so every platform computes the same permutation.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PLAAC_SHUF_FN __host__ __device__ __forceinline__
#else
#define PLAAC_SHUF_FN inline
#endif

namespace plaac {

constexpr int kShuffleRounds = 6;
constexpr uint64_t kShuffleGamma = 0x9E3779B97F4A7C15ull;

PLAAC_SHUF_FN uint64_t shuffle_mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

PLAAC_SHUF_FN uint32_t shuffle_mix32(uint32_t x)
{
    x ^= x >> 16;
    x *= 0x7feb352du;
    x ^= x >> 15;
    x *= 0x846ca68bu;
    x ^= x >> 16;
    return x;
}

// The permutation of one replicate: its domain width and round keys.
struct ShuffleKey {
    uint32_t key[kShuffleRounds];
    uint32_t n;  // protein length (< 2^31)
    int32_t b;   // domain bits; 0 for n <= 1
};

PLAAC_SHUF_FN ShuffleKey shuffle_key(uint64_t seed, int64_t protein, int64_t replicate, int64_t n)
{
    ShuffleKey k;
    uint64_t s = shuffle_mix64(seed + kShuffleGamma) ^ (uint64_t)protein;
    s = shuffle_mix64(s + kShuffleGamma) ^ (uint64_t)replicate;
    for (int r = 0; r < kShuffleRounds; r++) k.key[r] = (uint32_t)shuffle_mix64(s + (uint64_t)(r + 1) * kShuffleGamma);
    k.n = (uint32_t)n;
    int b = 0;
    while (b < 32 && n > 1 && ((uint64_t)(n - 1) >> b) != 0) b++;
    k.b = b;
    return k;
}

PLAAC_SHUF_FN uint32_t shuffle_feistel(const ShuffleKey& k, uint32_t x)
{
    const int b = k.b, lo = b >> 1, hi = b - lo;
#pragma unroll
    for (int r = 0; r < kShuffleRounds; r++) {
        const int w = (r & 1) ? hi : lo;  // bits of R; L has b - w
        const uint32_t R = x & ((1u << w) - 1u), L = x >> w;
        x = (R << (b - w)) | (L ^ (shuffle_mix32(R ^ k.key[r]) & ((1u << (b - w)) - 1u)));
    }
    return x;
}

// pi(t) for t < n.
PLAAC_SHUF_FN uint32_t shuffle_index(const ShuffleKey& k, uint32_t t)
{
    if (k.n <= 1) return t;
    do t = shuffle_feistel(k, t);
    while (t >= k.n);
    return t;
}

}  // namespace plaac

#undef PLAAC_SHUF_FN
