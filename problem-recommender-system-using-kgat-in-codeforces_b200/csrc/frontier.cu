// Needed-row frontier of a TRAIN_CF step (exact pruning of the propagation, reference model.py:165-202).
//
// The BPR loss gathers only the <= 3B batch rows of the propagated tables (model.py:189-191), so a row of layer l
// matters only if it is a batch row or a graph neighbour (through layers l+1 .. L) of one:
//     F_L = {batch ids},   F_{l-1} = F_l  U  cols(A[F_l, :])          (aggregator.py:54 reads E_{l-1}[c] for A[r, c] != 0)
// Everything outside F_l has an exactly-zero gradient and is never read, so layer l is computed (forward and
// backward) for the rows of F_l only -- same loss, same gradients as the reference's full propagation.
// A frontier level is a bitmap over the nodes (one bit per node, tested by the masked SpMM, spmm.cu) plus the
// ascending list of its rows (enumerated by the bi-interaction kernels).  All of it is stream-ordered device
// work with device-side counts, so a whole step still replays as one CUDA graph.
// Membership is collected in a BYTE-per-node flag array with plain stores (idempotent, so no atomics: 700 k edge
// visits at the Amazon-book shape would otherwise serialise on the ~160 cache lines of a 20 KB bitmap -- measured
// 98 us with atomicOr, see profiles/) and folded into the bitmap by the listing pass, which also clears the flags.
#include <stdlib.h>

#include "common.cuh"

namespace kgat {
namespace {

constexpr int kListBlock = 256;  // bitmap words per CTA of the listing kernels (one word per thread)

__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// flags[id] = 1; ids outside [0, n_nodes) are counted in *bad and skipped (the reference raises an IndexError)
__global__ void frontier_mark_kernel(const int64_t* __restrict__ ids, int64_t n_ids, int64_t n_nodes, uint8_t* __restrict__ flags,
                                     int32_t* __restrict__ bad) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_ids) return;
    const int64_t id = ids[i];
    if (id < 0 || id >= n_nodes) {
        if (bad != nullptr) atomicAdd(bad, 1);
        return;
    }
    flags[id] = 1;
}

// flags[r] = flags[c] = 1 for every listed row r and every column c of A[r, :].  Work items are the SpMM plan's tasks
// (<= chunk edges each, graph.py), enumerated like the row-list SpMM does: the chunk tasks of the heavy rows first
// (filtered by the level's bitmap), then one task per listed light row -- so a hub row does not serialise on one warp.
// Measured at the Amazon-book shape (tools/prof_frontier.py, ~35 k source rows; profiles/r2_frontier_variants.txt): testing a flag
// before setting it costs more than it saves -- the loads of a byte other SMs are storing to are slower than the redundant stores
// (test through L2, 32 edges at a time: 87 us; 256 at a time: 113 us; test through L1: 148 us; store without a test: 57 us; the
// shared-memory kernel below: 45 us).  This kernel is the fallback for graphs whose node bitmap does not fit in shared memory.
__global__ void __launch_bounds__(128) frontier_expand_kernel(const int4* __restrict__ tasks, int n_heavy_tasks,
                                                              const int32_t* __restrict__ light_rank, const int32_t* __restrict__ col_idx,
                                                              const int32_t* __restrict__ rows, const int32_t* __restrict__ cnt_dev,
                                                              const uint32_t* __restrict__ level_mask, uint8_t* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int n_warps = (gridDim.x * blockDim.x) >> 5;
    const int total = n_heavy_tasks + cnt_dev[0];
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < total; i += n_warps) {
        int4 t;
        if (i < n_heavy_tasks) {
            t = __ldg(tasks + i);
            if (!((__ldg(level_mask + (t.x >> 5)) >> (t.x & 31)) & 1u)) continue;
        } else {
            const int lr = __ldg(light_rank + __ldg(rows + (i - n_heavy_tasks)));
            if (lr < 0) continue;
            t = __ldg(tasks + n_heavy_tasks + lr);
        }
        if (lane == 0) flags[t.x] = 1;
        for (int base = t.y; base < t.z; base += 256) {
            int c[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int k = base + q * 32 + lane;
                c[q] = k < t.z ? __ldg(col_idx + k) : -1;
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (c[q] >= 0) flags[c[q]] = 1;
        }
    }
}

// Default: one persistent 1024-thread CTA per SM keeps a bitmap of the WHOLE node range in shared memory (n_nodes / 8 bytes); an edge's
// column goes to the global flag array only the first time this CTA sees it, so a hub column costs <= one global store per SM.
__global__ void __launch_bounds__(1024) frontier_expand_smem_kernel(const int4* __restrict__ tasks, int n_heavy_tasks,
                                                                    const int32_t* __restrict__ light_rank, const int32_t* __restrict__ col_idx,
                                                                    const int32_t* __restrict__ rows, const int32_t* __restrict__ cnt_dev,
                                                                    const uint32_t* __restrict__ level_mask, uint8_t* __restrict__ flags,
                                                                    int n_words) {
    extern __shared__ __align__(16) uint32_t seen_bits[];
    for (int w = threadIdx.x; w < n_words; w += 1024) seen_bits[w] = 0u;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int n_warps = (gridDim.x * 1024) >> 5;
    const int total = n_heavy_tasks + cnt_dev[0];
    // consecutive items to consecutive CTAs (not warps): the chunks of one hub row then meet different shared bitmaps, its columns
    // (mostly other hubs) are deduplicated against what the CTA's other 31 warps have already seen
    for (int i = blockIdx.x + gridDim.x * (threadIdx.x >> 5); i < total; i += n_warps) {
        int4 t;
        if (i < n_heavy_tasks) {
            t = __ldg(tasks + i);
            if (!((__ldg(level_mask + (t.x >> 5)) >> (t.x & 31)) & 1u)) continue;
        } else {
            const int lr = __ldg(light_rank + __ldg(rows + (i - n_heavy_tasks)));
            if (lr < 0) continue;
            t = __ldg(tasks + n_heavy_tasks + lr);
        }
        if (lane == 0) flags[t.x] = 1;
        for (int base = t.y; base < t.z; base += 256) {
            int c[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int k = base + q * 32 + lane;
                c[q] = k < t.z ? __ldg(col_idx + k) : -1;
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                if (c[q] < 0) continue;
                const uint32_t bit = 1u << (c[q] & 31);
                if (seen_bits[c[q] >> 5] & bit) continue;
                if (!(atomicOr(seen_bits + (c[q] >> 5), bit) & bit)) flags[c[q]] = 1;
            }
        }
    }
}

// bitmap word w <- flags[32 w .. 32 w + 32) (and the flags are cleared for the next build); block totals of the set bits
__global__ void __launch_bounds__(kListBlock) frontier_count_kernel(uint8_t* __restrict__ flags, uint32_t* __restrict__ bitmap,
                                                                   int64_t n_words, int32_t* __restrict__ block_total) {
    __shared__ int sh[kListBlock / 32];
    const int64_t w = blockIdx.x * (int64_t)kListBlock + threadIdx.x;
    int c = 0;
    if (w < n_words) {
        uint4* f4 = reinterpret_cast<uint4*>(flags + w * 32);
        const uint4 a = f4[0], b = f4[1];
        const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t bits = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            // byte j of v[q] non-zero -> bit 4 q + j
            const uint32_t x = v[q];
            bits |= ((x & 0xffu) ? 1u : 0u) << (4 * q) | ((x & 0xff00u) ? 1u : 0u) << (4 * q + 1) | ((x & 0xff0000u) ? 1u : 0u) << (4 * q + 2) |
                    ((x & 0xff000000u) ? 1u : 0u) << (4 * q + 3);
        }
        bitmap[w] = bits;
        if (bits) {
            f4[0] = make_uint4(0u, 0u, 0u, 0u);
            f4[1] = make_uint4(0u, 0u, 0u, 0u);
        }
        c = __popc(bits);
    }
    c = warp_sum_i(c);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < kListBlock / 32; ++i) t += sh[i];
        block_total[blockIdx.x] = t;
    }
}

// rows[...] = ascending node ids of the set bits; *cnt = their number
__global__ void __launch_bounds__(kListBlock) frontier_write_kernel(const uint32_t* __restrict__ bitmap, int64_t n_words,
                                                                   const int32_t* __restrict__ block_total, int32_t* __restrict__ rows,
                                                                   int32_t* __restrict__ cnt) {
    __shared__ int sh[kListBlock / 32];
    __shared__ int sh_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // rows of all earlier blocks
    int part = 0;
    for (int j = tid; j < (int)blockIdx.x; j += kListBlock) part += block_total[j];
    part = warp_sum_i(part);
    if (lane == 0) sh[warp] = part;
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int i = 0; i < kListBlock / 32; ++i) t += sh[i];
        sh_base = t;
    }
    __syncthreads();
    const int base = sh_base;
    __syncthreads();
    const int64_t w = blockIdx.x * (int64_t)kListBlock + tid;
    uint32_t bits = w < n_words ? bitmap[w] : 0u;
    const int c = __popc(bits);
    int incl = c;  // inclusive scan inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) sh[warp] = incl;
    __syncthreads();
    int woff = 0;
    for (int i = 0; i < warp; ++i) woff += sh[i];
    int pos = base + woff + incl - c;
    while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        rows[pos++] = (int)(w * 32 + b);
    }
    if (blockIdx.x == gridDim.x - 1 && tid == kListBlock - 1) cnt[0] = pos;  // the last thread ends at the grand total
}

// T[rows[i], :] = 0 for i < *cnt  (the gradient rows of the last table, before the BPR scatter)
__global__ void frontier_zero_rows_kernel(float* __restrict__ T, int64_t ld, int d4, const int32_t* __restrict__ rows,
                                          const int32_t* __restrict__ cnt_dev) {
    const int cnt = cnt_dev[0];
    const int64_t total = (int64_t)cnt * d4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = rows[i / d4];
        reinterpret_cast<float4*>(T + (int64_t)r * ld)[i % d4] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// The part of a level that falls into a node range [lo, hi) (both multiples of 32): its rows -- a contiguous segment of the
// ascending list -- and its bitmap words.  Row-sharded multi-GPU runs compute a layer for "level AND my range".
__global__ void __launch_bounds__(256) frontier_segment_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ cnt_dev,
                                                               const uint32_t* __restrict__ mask, int lo, int hi, int n_words,
                                                               int32_t* __restrict__ out_rows, int32_t* __restrict__ out_cnt,
                                                               uint32_t* __restrict__ out_mask) {
    __shared__ int seg[2];
    if (threadIdx.x < 2) {  // first list position holding a row >= lo (thread 0) / >= hi (thread 1)
        const int key = threadIdx.x == 0 ? lo : hi;
        int a = 0, b = cnt_dev[0];
        while (a < b) {
            const int m = (a + b) >> 1;
            if (rows[m] < key) a = m + 1; else b = m;
        }
        seg[threadIdx.x] = a;
    }
    __syncthreads();
    const int begin = seg[0], n = seg[1] - seg[0];
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    for (int i = tid; i < n; i += stride) out_rows[i] = rows[begin + i];
    for (int w = tid; w < n_words; w += stride) out_mask[w] = (w >= (lo >> 5) && w < (hi >> 5)) ? mask[w] : 0u;
    if (tid == 0) out_cnt[0] = n;
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int kgat_frontier_segment(const int32_t* rows, const int32_t* count_dev, const uint32_t* bitmap, int64_t n_nodes, int64_t lo, int64_t hi,
                          int32_t* out_rows, int32_t* out_count_dev, uint32_t* out_bitmap, void* stream) {
    if (!rows || !count_dev || !bitmap || !out_rows || !out_count_dev || !out_bitmap || n_nodes <= 0 || lo < 0 || hi < lo || (lo & 31) ||
        ((hi & 31) && hi != n_nodes) || hi > ((n_nodes + 31) / 32) * 32 || n_nodes >= ((int64_t)1 << 31))
        return KGAT_ERR_INVALID_ARGUMENT;
    const int n_words = (int)((n_nodes + 31) / 32);
    const int64_t hi_w = (hi + 31) / 32 * 32;  // the last range may end at n_nodes: its final word is whole anyway (no bits beyond n)
    int ctas = (int)(((hi - lo) + 255) / 256);
    if (ctas < 1) ctas = 1;
    if (ctas > sm_count()) ctas = sm_count();
    frontier_segment_kernel<<<ctas, 256, 0, (cudaStream_t)stream>>>(rows, count_dev, bitmap, (int)lo, (int)hi_w, n_words, out_rows, out_count_dev,
                                                                   out_bitmap);
    return check_launch();
}

int64_t kgat_frontier_scratch_ints(int64_t n_nodes) {
    const int64_t n_words = (n_nodes + 31) / 32;
    return (n_words + kListBlock - 1) / kListBlock + 1;
}

int kgat_frontier_mark_ids(const int64_t* ids64, int64_t n_ids, int64_t n_nodes, uint8_t* flags, int32_t* bad_count_dev, void* stream) {
    if (n_ids < 0 || n_nodes <= 0 || !flags) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_ids == 0) return KGAT_OK;
    frontier_mark_kernel<<<(unsigned)((n_ids + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ids64, n_ids, n_nodes, flags, bad_count_dev);
    return check_launch();
}

int kgat_frontier_expand(const int32_t* tasks, int64_t n_heavy_tasks, const int32_t* light_rank, const int32_t* col_idx,
                         const int32_t* rows, const int32_t* count_dev, int64_t max_rows, const uint32_t* level_bitmap, uint8_t* flags,
                         int64_t n_nodes, void* stream) {
    if (!tasks || !light_rank || !col_idx || !rows || !count_dev || !flags || max_rows <= 0 || n_heavy_tasks < 0 || n_nodes <= 0 ||
        (n_heavy_tasks > 0 && !level_bitmap) || n_heavy_tasks >= ((int64_t)1 << 30))
        return KGAT_ERR_INVALID_ARGUMENT;
    int64_t ctas = (max_rows + n_heavy_tasks + 3) / 4;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (ctas > cap) ctas = cap;
    static const bool plain = [] {  // KGAT_EXPAND_PLAIN=1: the global-store kernel even when the bitmap fits (A/B, tools/prof_frontier.py)
        const char* e = getenv("KGAT_EXPAND_PLAIN");
        return e && atoi(e) == 1;
    }();
    const int4* t4 = reinterpret_cast<const int4*>(tasks);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n_words = (n_nodes + 31) / 32;
    if (!plain && n_words * 4 <= 200 * 1024) {
        static uint64_t configured = 0;
        if (const int rc = raise_smem_limit(frontier_expand_smem_kernel, 200 * 1024, configured); rc != KGAT_OK) return rc;
        int64_t big = (max_rows + n_heavy_tasks + 31) / 32;
        if (big > sm_count()) big = sm_count();
        frontier_expand_smem_kernel<<<(unsigned)big, 1024, (size_t)n_words * 4, st>>>(t4, (int)n_heavy_tasks, light_rank, col_idx, rows, count_dev,
                                                                                     level_bitmap, flags, (int)n_words);
        return check_launch();
    }
    frontier_expand_kernel<<<(unsigned)ctas, 128, 0, st>>>(t4, (int)n_heavy_tasks, light_rank, col_idx, rows, count_dev, level_bitmap, flags);
    return check_launch();
}

int kgat_frontier_list(uint8_t* flags, uint32_t* bitmap, int64_t n_nodes, int32_t* scratch, int32_t* rows, int32_t* count_dev, void* stream) {
    if (!flags || !bitmap || !scratch || !rows || !count_dev || n_nodes <= 0 || n_nodes >= ((int64_t)1 << 31)) return KGAT_ERR_INVALID_ARGUMENT;
    if (reinterpret_cast<uintptr_t>(flags) & 15) return KGAT_ERR_INVALID_ARGUMENT;
    const int64_t n_words = (n_nodes + 31) / 32;
    const unsigned blocks = (unsigned)((n_words + kListBlock - 1) / kListBlock);
    frontier_count_kernel<<<blocks, kListBlock, 0, (cudaStream_t)stream>>>(flags, bitmap, n_words, scratch);
    frontier_write_kernel<<<blocks, kListBlock, 0, (cudaStream_t)stream>>>(bitmap, n_words, scratch, rows, count_dev);
    return check_launch();
}

int kgat_frontier_zero_rows(float* T, int64_t ld, int32_t d, const int32_t* rows, const int32_t* count_dev, int64_t max_rows, void* stream) {
    if (!T || !rows || !count_dev || d <= 0 || (d & 3) || (ld & 3) || max_rows <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    int64_t ctas = (max_rows * (d / 4) + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 4;
    if (ctas > cap) ctas = cap;
    frontier_zero_rows_kernel<<<(unsigned)ctas, 256, 0, (cudaStream_t)stream>>>(T, ld, d / 4, rows, count_dev);
    return check_launch();
}

}  // extern "C"
