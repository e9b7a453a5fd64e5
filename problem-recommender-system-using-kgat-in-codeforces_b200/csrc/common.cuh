// Shared device/host helpers for libkgat_b200 (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kgat_b200.h"

#define KGAT_LEAKY_SLOPE 0.01f  // nn.LeakyReLU() default (reference aggregator.py:23)
#define KGAT_NORM_EPS 1e-12f    // F.normalize default eps (reference aggregator.py:65)

namespace kgat {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// thread-local record of the last CUDA failure (kgat_last_cuda_error)
void set_cuda_error(cudaError_t e);

inline int check_launch() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_cuda_error(e);
        return KGAT_ERR_CUDA;
    }
    return KGAT_OK;
}

inline int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            n <= 0)
            n = 148;  // B200
    }
    return n;
}

#define KGAT_CUDA_TRY(expr)                  \
    do {                                     \
        cudaError_t e__ = (expr);            \
        if (e__ != cudaSuccess) {            \
            ::kgat::set_cuda_error(e__);     \
            return KGAT_ERR_CUDA;            \
        }                                    \
    } while (0)

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
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

// read-only 128-bit gather (L1-allocating: hub rows are re-read by neighbouring warps)
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// streaming 128-bit load that does not pollute L1
__device__ __forceinline__ float4 ld_stream4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void fma4(float4& a, float s, const float4& x) {
    a.x = fmaf(s, x.x, a.x);
    a.y = fmaf(s, x.y, a.y);
    a.z = fmaf(s, x.z, a.z);
    a.w = fmaf(s, x.w, a.w);
}
__device__ __forceinline__ float lrelu(float z) { return z > 0.f ? z : KGAT_LEAKY_SLOPE * z; }

// order-preserving map: larger float -> larger key; -inf smallest; NaN treated as largest (torch.sort)
__device__ __forceinline__ uint32_t float_key(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// first position in p[0, n) whose value is >= x (p ascending)
__device__ __forceinline__ int lower_bound_i32(const int32_t* __restrict__ p, int n, int x) {
    int lo = 0;
    while (n > 0) {
        const int half = n >> 1;
        if (__ldg(p + lo + half) < x) {
            lo += half + 1;
            n -= half + 1;
        } else {
            n = half;
        }
    }
    return lo;
}

// kgat_tables_t in float4 units: table t holds columns [4 qoff[t], 4 qoff[t+1]) of the concatenated row
struct ConcatTables {
    int n;
    int q[KGAT_MAX_LAYERS];
    int qoff[KGAT_MAX_LAYERS + 1];
    const float* p[KGAT_MAX_LAYERS];
    int64_t ld[KGAT_MAX_LAYERS];
};

// false when a table is missing or a width / leading dimension is not a multiple of 4
inline bool tables_from(const kgat_tables_t* t, ConcatTables* T) {
    if (!t || t->n_tables <= 0 || t->n_tables > KGAT_MAX_LAYERS) return false;
    T->n = t->n_tables;
    T->qoff[0] = 0;
    for (int i = 0; i < T->n; ++i) {
        if (t->dims[i] <= 0 || (t->dims[i] & 3) || (t->lds[i] & 3) || !t->tables[i]) return false;
        T->q[i] = t->dims[i] / 4;
        T->qoff[i + 1] = T->qoff[i] + T->q[i];
        T->p[i] = t->tables[i];
        T->ld[i] = t->lds[i];
    }
    return true;
}

// log(sigmoid(x)) as ATen computes it: min(x,0) - log1p(exp(-|x|))
__device__ __forceinline__ float log_sigmoid(float x) { return fminf(x, 0.f) - log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// ------------------------------------------------------------------------------------------
// Philox4x32-10 counter RNG (dropout decisions).  One call gives 4 x 32 random bits for a
// (seed, counter) pair; the stream is a pure function of its arguments so the backward pass or
// a CUDA-graph replay can regenerate it without storing state.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint64_t seed, uint64_t counter) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)counter, c1 = (uint32_t)(counter >> 32), c2 = 0x4b474154u /* "KGAT" */, c3 = 0u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    return make_uint4(c0, c1, c2, c3);
}
// uniform in [0,1) from 32 bits (24-bit mantissa path)
__device__ __forceinline__ float u01(uint32_t bits) { return (bits >> 8) * (1.0f / 16777216.0f); }

}  // namespace kgat
