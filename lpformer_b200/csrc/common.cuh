// Shared helpers for the lpformer_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/lpformer_b200.h"

namespace lpf {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kNumSMs = 148;  // B200

void set_error(const char* fmt, ...);

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return LPF_ERR_CUDA;
    }
    return LPF_OK;
}

#define LPF_REQUIRE(cond, msg)                                  \
    do {                                                        \
        if (!(cond)) {                                          \
            lpf::set_error("%s: %s", __func__, msg);            \
            return LPF_ERR_INVALID;                             \
        }                                                       \
    } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// q(p) = fl32(p + 1) - 1: the fp32 round trip the reference applies to every PPR value
// before thresholding (models/link_transformer.py:290-291,316-317,464-476).  Must not be
// contracted or reassociated, hence the explicit round-to-nearest intrinsics.
__device__ __forceinline__ float quantise(float p) { return __fsub_rn(__fadd_rn(p, 1.0f), 1.0f); }

// ---------------------------------------------------------------------------------------------------------- dropout
// Counter-based random numbers of every dropout site (the rule of include/lpformer_b200.h, "Dropout"): Philox4x32-10
// (Salmon et al., SC'11) with key = the 64-bit seed (low word, high word) and counter = (col >> 2, row low word, row
// high word, site).  Element (row, col) reads word (col & 3) of the block, so a mask is a pure function of
// (seed, site, row, col): independent of launch shape, row sharding and index subsets.  The element is kept iff that
// word u satisfies u >= thr with thr = floor(p 2^32) (p = 0 keeps every element, p = 1 none), and a kept element is
// multiplied by scale = fp32(1 / (1 - p)); a dropped one becomes 0.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    }
    return c;
}

// the four words of columns [4 group, 4 group + 4) of `row`
__device__ __forceinline__ uint4 dropout_bits(uint64_t seed, int site, int64_t row, int64_t group) {
    return philox4x32_10(make_uint4((uint32_t)group, (uint32_t)(uint64_t)row, (uint32_t)((uint64_t)row >> 32), (uint32_t)site),
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}

__device__ __forceinline__ uint32_t uint4_word(uint4 u, int j) {
    return j == 0 ? u.x : j == 1 ? u.y : j == 2 ? u.z : u.w;
}

// x kept (x * scale) or dropped (0) by word u
__device__ __forceinline__ float dropout_apply(float x, uint32_t u, uint64_t thr, float scale) {
    return (uint64_t)u >= thr ? x * scale : 0.f;
}

// thr and scale of the keep rule for probability p; false when p is outside [0, 1]
inline bool dropout_rule(double p, uint64_t* thr, float* scale) {
    if (!(p >= 0.0 && p <= 1.0)) return false;
    *thr = (uint64_t)(p * 4294967296.0);           // (exact: p * 2^32 only shifts the exponent; the cast floors)
    *scale = p < 1.0 ? (float)(1.0 / (1.0 - p)) : 0.f;
    return true;
}

// lower_bound over a sorted int32 row in global memory.
__device__ __forceinline__ int lower_bound(const int32_t* __restrict__ a, int n, int32_t key) {
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (__ldg(a + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

}  // namespace lpf
