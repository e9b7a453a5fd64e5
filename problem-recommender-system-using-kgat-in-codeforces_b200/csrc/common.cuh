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

inline int padded_width(const ConcatTables& T) { return ((T.qoff[T.n] * 4 + 15) / 16) * 16; }

// float4 of concatenated columns [4 q, 4 q + 4) of table row `id` (zeros past the width)
__device__ __forceinline__ float4 concat_quad(const ConcatTables& T, int64_t id, int q) {
    int t = 0;
    while (t < T.n && q >= T.qoff[t + 1]) ++t;
    if (t == T.n) return make_float4(0.f, 0.f, 0.f, 0.f);
    return ldg4(T.p[t] + id * T.ld[t] + (q - T.qoff[t]) * 4);
}

// ------------------------------------------------------------------------------------------
// 64-user x 64-candidate score tiles of the fused scoring kernels (recommend.cu, rank.cu): 256 threads, thread (tx, ty) =
// (tid % 16, tid / 16) owns users ty * 4 + i and candidates tx * 4 + j of a tile.  The arithmetic is sgemm_nt_kernel's:
// a sequential fmaf chain from +0 over the concatenated columns in ascending order, zero-padded to a multiple of 16.
// ------------------------------------------------------------------------------------------
constexpr int kTileThreads = 256;
constexpr int kTileUsers = 64;
constexpr int kTileItems = 64;
constexpr int kTilePad = 68;       // shared row stride (floats) of the transposed tiles, as in sgemm_nt_kernel
constexpr int kTileMaxSlices = 64;

// shared floats of the user tile [width_pad][kTilePad] and the candidate slab [16][kTilePad]
inline size_t tile_smem_floats(int width_pad) { return (size_t)(width_pad + 16) * kTilePad; }

// Us[c][r] = column c of users[u0 + r]'s concatenated row (zero rows past n_users).  The caller synchronises afterwards.
__device__ __forceinline__ void stage_user_tile(const ConcatTables& T, const int32_t* __restrict__ users, int n_users, int u0, int width_pad,
                                                float* Us) {
    const int nq = width_pad / 4;
    for (int e = threadIdx.x; e < kTileUsers * nq; e += kTileThreads) {
        const int r = e % kTileUsers, q = e / kTileUsers;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (u0 + r < n_users) v = concat_quad(T, users[u0 + r], q);
        Us[(4 * q + 0) * kTilePad + r] = v.x;
        Us[(4 * q + 1) * kTilePad + r] = v.y;
        Us[(4 * q + 2) * kTilePad + r] = v.z;
        Us[(4 * q + 3) * kTilePad + r] = v.w;
    }
}

// acc[i][j] = score of staged user ty * 4 + i and candidate c0 + tx * 4 + j (candidates from c_end on score 0).  Every thread
// of the CTA calls it; it synchronises before each write of the slab Bs, so the caller may read acc without a barrier.
__device__ __forceinline__ void score_tile(const ConcatTables& T, const int32_t* __restrict__ cand, int c0, int c_end, int width_pad, const float* Us,
                                           float* Bs, float (&acc)[4][4]) {
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const int lr = tid / 4, lk = (tid % 4) * 4;  // slab load mapping: 64 candidates x 16 columns, one float4 per thread
    const int my_c = c0 + lr;
    const int64_t my_id = my_c < c_end ? cand[my_c] : -1;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < width_pad; k0 += 16) {
        const float4 b = my_id >= 0 ? concat_quad(T, my_id, (k0 + lk) / 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();
        Bs[(lk + 0) * kTilePad + lr] = b.x;
        Bs[(lk + 1) * kTilePad + lr] = b.y;
        Bs[(lk + 2) * kTilePad + lr] = b.z;
        Bs[(lk + 3) * kTilePad + lr] = b.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(&Us[(k0 + kk) * kTilePad + ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk * kTilePad + tx * 4]);
            const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
        }
    }
}

// candidate slices per 64-user tile: enough CTAs for two waves over the SMs while the users alone do not give them (per_sm =
// resident CTAs per SM of the kernel), at least one 64-candidate tile per slice; `requested` > 0 is taken as is
inline int pick_slices(int64_t n_users, int64_t n_cand_max, int per_sm, int requested) {
    if (requested > 0) return requested;
    const int64_t tiles = (n_users + kTileUsers - 1) / kTileUsers;
    const int64_t want = 2LL * sm_count() * per_sm;
    int64_t s = tiles > 0 ? (want + tiles - 1) / tiles : 1;
    const int64_t by_items = (n_cand_max + kTileItems - 1) / kTileItems;
    if (s > by_items) s = by_items;
    if (s > kTileMaxSlices) s = kTileMaxSlices;
    return (int)(s < 1 ? 1 : s);
}

// ------------------------------------------------------------------------------------------
// Running top-k lists of the fused selection kernels (recommend.cu, complete.cu): an entry is a value and a candidate index,
// ordered by descending float_key(value), then ascending index -- a total order, so a list does not depend on how the
// candidates were split.  k <= kTopkMaxK; a CTA folds at most kTileItems pending entries per row at a time.
// ------------------------------------------------------------------------------------------
constexpr int kTopkMaxK = 128;  // = kTopkMax of topk_rows

struct Entry {
    float s;
    int c;  // candidate index
};

// true when a ranks before b
__device__ __forceinline__ bool beats(const Entry& a, const Entry& b) {
    const uint32_t ka = float_key(a.s), kb = float_key(b.s);
    return ka != kb ? ka > kb : a.c < b.c;
}

// number of entries of the sorted list l[0, n) that beat x
__device__ __forceinline__ int count_beating(const Entry* l, int n, const Entry& x) {
    int lo = 0;
    while (n > 0) {
        const int half = n >> 1;
        if (beats(l[lo + half], x)) {
            lo += half + 1;
            n -= half + 1;
        } else {
            n = half;
        }
    }
    return lo;
}

// One warp folds the np <= kTileItems unordered entries pl into the sorted list tl[0, nt): rank = members of the union that
// beat it.  Returns the new length min(nt + np, k).
__device__ __forceinline__ int fold_pending(Entry* tl, int nt, const Entry* pl, int np, int k, int lane) {
    constexpr int M = (kTopkMaxK + kTileItems) / 32;
    const int n_union = nt + np;
    Entry xs[M];
    int rk[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        const int e = lane + 32 * m;
        rk[m] = k;
        if (e < n_union) {
            const Entry x = e < nt ? tl[e] : pl[e - nt];
            int r = e < nt ? e : count_beating(tl, nt, x);
            for (int j = 0; j < np && r < k; ++j) r += beats(pl[j], x);
            xs[m] = x;
            rk[m] = r;
        }
    }
    __syncwarp();
#pragma unroll
    for (int m = 0; m < M; ++m)
        if (rk[m] < k) tl[rk[m]] = xs[m];
    __syncwarp();
    return n_union < k ? n_union : k;
}

// One warp merges a row's per-slice sorted lists (lists[s * k ..], lens[s]) by rank: put(r, x) for every entry x of merged
// rank r < k.  Returns min(k, total entries).
template <class Put>
__device__ __forceinline__ int merge_slices(const Entry* lists, const int32_t* lens, int slices, int k, int lane, Put put) {
    int total = 0;
    for (int s = 0; s < slices; ++s) total += lens[s];
    for (int e = lane; e < slices * k; e += 32) {
        const int s = e / k, i = e % k;
        if (i >= lens[s]) continue;
        const Entry x = lists[e];
        int r = i;
        for (int v = 0; v < slices && r < k; ++v)
            if (v != s) r += count_beating(lists + v * k, lens[v], x);
        if (r < k) put(r, x);
    }
    return total < k ? total : k;
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
