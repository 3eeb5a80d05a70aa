// Shared device-side definitions for libplaac_cuda.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/plaac_cuda.h"

namespace plaac {

constexpr int kPad = 22;          // pad code: every table entry is 0 for it
constexpr int kPapaMaskBit = 32;  // ext code bit: "proline not scored by PAPA" (plaac.java:2652-2655)
constexpr int kTabN = 64;         // per-code tables are indexed by ext code 0..63
constexpr int kChunk = 16;        // residues per 16-byte lane slot
constexpr int kHistBins = 32768;  // exact-length bins; longer proteins share bin 0

// Scalars of plaac_params the kernels read straight from the constant bank (kernel argument).
struct KScalars {
    int32_t core_len, w, h_fi, h_papa, mw_window, adjust_prolines;
    uint32_t charge_plus, charge_minus, qn_mask;
    double lt00, lt01, lt10, lt11, li0, li1, lf0, lf1;
    double cc0, cc1, cc2, big_neg, ln2;
};

// Per-code tables + LUT as uploaded once per ctx (global memory; kernels stage them in shared memory).
struct DeviceTables {
    double le0[kTabN], le1[kTabN], lebg[kTabN], llr[kTabN], hyd[kTabN], pap[kTabN];
    // hydropathy rounded to the 2^-k grid on which every window sum of up to (2w+2)^2 taps is exact (like pap): the
    // sliding-window sums of the summary kernels are then exact, i.e. independent of the order and of where a running
    // sum was (re)started; hyd stays exact for the sequential mean and the per-residue tracks
    double hydw[kTabN];
    // hydw[e] ~ hydi[e] / q when the host proved the integer form of the FoldIndex tests exact (plan_int_fold), else 0
    int32_t hydi[kTabN];
    double lut[PLAAC_LUT_LEN + 3];
};

// Work description of one device batch after bucketing.
struct BatchView {
    const uint4* stream;      // [slot][lane] ext codes, 16 per slot; slot = chunk_base[b] + j
    uint32_t* tbw;            // same indexing, one word per slot: traceback bits, later Viterbi bits
    const int32_t* order;     // sorted rank -> protein index (descending length)
    const int64_t* offsets;   // nprot+1
    const int64_t* chunk_base;  // nbuckets+1, in slots-of-32-lanes
    const int32_t* slot_bucket; // bucket of every 32-lane slot (written by k_pack)
    int64_t nslots;           // chunk_base[nbuckets] if the host knows it, else an upper bound
    int64_t nprot;
    int64_t nbuckets;
    int64_t off_base;         // offsets[] are relative to this residue index
    int64_t long_min;         // proteins at least this long belong to the long-sequence path: empty for the bucketed one
};

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the FUNCTION on the device, shared by every ctx of the process:
// it is raised once to everything the device allows (opt-in maximum minus the kernel's static shared memory), never to one
// ctx's own sizes -- a ctx created later with smaller rings would otherwise lower the limit under an earlier ctx.
inline cudaError_t raise_dynamic_smem_limit(const void* fn, int optin_bytes, size_t need_bytes)
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, fn);
    if (e != cudaSuccess) return e;
    const long long room = (long long)optin_bytes - (long long)a.sharedSizeBytes;
    if (room < (long long)need_bytes) return cudaErrorInvalidValue;
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)room);
}

// Length of a protein as the bucketed path sees it.
__device__ __forceinline__ int64_t eff_len(int64_t len, int64_t long_min) { return len >= long_min ? 0 : len; }

}  // namespace plaac
