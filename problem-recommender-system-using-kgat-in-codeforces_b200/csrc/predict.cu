// K9/K10: predict path.  Gather the concatenated layer rows of users / items, score GEMM
// (reference model.py:388-391), train-positive masking and descending top-K with the CPU
// torch.sort tie order (reference metrics_calculator.py:118-121, main.py:592-604).
#include "common.cuh"

namespace kgat {
namespace {

__global__ void __launch_bounds__(256) gather_concat_kernel(ConcatTables T, const int64_t* __restrict__ ids, int64_t n_ids,
                                                            float* __restrict__ out, int64_t ld_out) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (b >= n_ids) return;
    const int64_t id = ids[b];
    for (int t = 0; t < T.n; ++t)
        for (int f = lane; f < T.q[t]; f += 32)
            *reinterpret_cast<float4*>(out + b * ld_out + (T.qoff[t] + f) * 4) = ldg4(T.p[t] + id * T.ld[t] + f * 4);
}

// C = A * B^T, 64x64 tile, BK = 16, 256 threads, 4x4 micro-tile (fp32 FMA)
__global__ void __launch_bounds__(256) sgemm_nt_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb,
                                                       float* __restrict__ C, int64_t ldc, int m, int n, int k) {
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;
    const int row0 = blockIdx.y * 64, col0 = blockIdx.x * 64;
    float acc[4][4] = {};
    const int lr = tid / 4, lk = (tid % 4) * 4;  // load mapping: 64 rows x 16 k, one float4 per thread
    for (int k0 = 0; k0 < k; k0 += 16) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        const bool kfull = k0 + lk + 3 < k;
        if (row0 + lr < m) {
            const float* src = A + (int64_t)(row0 + lr) * lda + k0 + lk;
            if (kfull && ((lda & 3) == 0)) a = ldg4(src);
            else { a.x = k0 + lk < k ? src[0] : 0.f; a.y = k0 + lk + 1 < k ? src[1] : 0.f; a.z = k0 + lk + 2 < k ? src[2] : 0.f; a.w = k0 + lk + 3 < k ? src[3] : 0.f; }
        }
        if (col0 + lr < n) {
            const float* src = B + (int64_t)(col0 + lr) * ldb + k0 + lk;
            if (kfull && ((ldb & 3) == 0)) b = ldg4(src);
            else { b.x = k0 + lk < k ? src[0] : 0.f; b.y = k0 + lk + 1 < k ? src[1] : 0.f; b.z = k0 + lk + 2 < k ? src[2] : 0.f; b.w = k0 + lk + 3 < k ? src[3] : 0.f; }
        }
        __syncthreads();
        As[lk + 0][lr] = a.x; As[lk + 1][lr] = a.y; As[lk + 2][lr] = a.z; As[lk + 3][lr] = a.w;
        Bs[lk + 0][lr] = b.x; Bs[lk + 1][lr] = b.y; Bs[lk + 2][lr] = b.z; Bs[lk + 3][lr] = b.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = row0 + ty * 4 + i;
        if (r >= m) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = col0 + tx * 4 + j;
            if (c < n) C[(int64_t)r * ldc + c] = acc[i][j];
        }
    }
}

__global__ void mask_scores_kernel(float* __restrict__ scores, int64_t ld, int m, int n, const int32_t* __restrict__ mask_ptr,
                                   const int32_t* __restrict__ mask_items) {
    const int row = blockIdx.x;
    if (row >= m) return;
    for (int p = mask_ptr[row] + threadIdx.x; p < mask_ptr[row + 1]; p += blockDim.x) {
        const int c = mask_items[p];
        if (c >= 0 && c < n) scores[(int64_t)row * ld + c] = -INFINITY;
    }
}

// Exact top-K of one row per CTA via 3-pass radix select on the 32-bit key, then an ordered
// collect (ties at the threshold are taken lowest-column-first) and a small sort of the K winners.
constexpr int kTopkThreads = 512;
constexpr int kTopkMax = 128;
__global__ void __launch_bounds__(kTopkThreads) topk_rows_kernel(const float* __restrict__ scores, int64_t ld, int m, int n, int k,
                                                                 int32_t* __restrict__ idx_out, float* __restrict__ val_out) {
    __shared__ int hist[2048];
    __shared__ uint32_t s_prefix, s_mask;
    __shared__ int s_need, s_count_gt, s_eq_base, s_warp_eq[kTopkThreads / 32];
    __shared__ uint32_t c_key[kTopkMax];
    __shared__ int c_idx[kTopkMax];
    const int row = blockIdx.x;
    const float* x = scores + (int64_t)row * ld;
    const int tid = threadIdx.x;
    if (tid == 0) { s_prefix = 0; s_mask = 0; s_need = k; }
    __syncthreads();
    const int shifts[3] = {21, 10, 0};
    const int widths[3] = {11, 11, 10};
    for (int pass = 0; pass < 3; ++pass) {
        const int nb = 1 << widths[pass];
        for (int i = tid; i < nb; i += kTopkThreads) hist[i] = 0;
        __syncthreads();
        const uint32_t prefix = s_prefix, mask = s_mask;
        for (int i = tid; i < n; i += kTopkThreads) {
            const uint32_t key = float_key(x[i]);
            if ((key & mask) == prefix) atomicAdd(&hist[(key >> shifts[pass]) & (nb - 1)], 1);
        }
        __syncthreads();
        if (tid == 0) {  // walk bins from the largest key downwards
            int need = s_need, b = nb - 1;
            for (; b > 0; --b) {
                if (hist[b] >= need) break;
                need -= hist[b];
            }
            s_need = need;  // how many still to take inside bin b
            s_prefix = prefix | ((uint32_t)b << shifts[pass]);
            s_mask = mask | ((uint32_t)(nb - 1) << shifts[pass]);
        }
        __syncthreads();
    }
    const uint32_t thr = s_prefix;  // exact key of the k-th largest element
    const int need_eq = s_need;     // number of elements == thr to take (lowest columns first)
    if (tid == 0) { s_count_gt = 0; s_eq_base = 0; }
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5;
    for (int base = 0; base < n; base += kTopkThreads) {
        const int i = base + tid;
        uint32_t key = 0;
        bool gt = false, eq = false;
        if (i < n) {
            key = float_key(x[i]);
            gt = key > thr;
            eq = key == thr;
        }
        if (gt) {
            const int pos = atomicAdd(&s_count_gt, 1);
            c_key[pos] = key;
            c_idx[pos] = i;
        }
        // ordered compaction of the == thr elements
        const unsigned bal = __ballot_sync(kFull, eq);
        if (lane == 0) s_warp_eq[warp] = __popc(bal);
        __syncthreads();
        if (eq) {
            int before = s_eq_base + __popc(bal & ((1u << lane) - 1));
            for (int w = 0; w < warp; ++w) before += s_warp_eq[w];
            if (before < need_eq) {
                const int pos = k - need_eq + before;  // the > thr winners occupy [0, k - need_eq)
                c_key[pos] = key;
                c_idx[pos] = i;
            }
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < kTopkThreads / 32; ++w) tot += s_warp_eq[w];
            s_eq_base += tot;
        }
        __syncthreads();
    }
    // rank sort of the k winners: descending key, ascending column on ties
    if (tid < k) {
        const uint32_t key = c_key[tid];
        const int id = c_idx[tid];
        int rank = 0;
        for (int j = 0; j < k; ++j) {
            const uint32_t kj = c_key[j];
            const int ij = c_idx[j];
            rank += (kj > key) || (kj == key && ij < id);
        }
        idx_out[(int64_t)row * k + rank] = id;
        if (val_out != nullptr) val_out[(int64_t)row * k + rank] = x[id];
    }
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int kgat_gather_concat(const kgat_tables_t* t, const int64_t* ids64, int64_t n_ids, float* out, int64_t ld_out, void* stream) {
    if (!t || t->n_tables <= 0 || t->n_tables > KGAT_MAX_LAYERS || n_ids < 0 || (ld_out & 3)) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_ids == 0) return KGAT_OK;
    ConcatTables T;
    if (!tables_from(t, &T)) return KGAT_ERR_INVALID_ARGUMENT;
    gather_concat_kernel<<<(unsigned)((n_ids * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(T, ids64, n_ids, out, ld_out);
    return check_launch();
}

int kgat_sgemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int32_t m, int32_t n, int32_t k,
                  void* stream) {
    if (m < 0 || n < 0 || k <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (m == 0 || n == 0) return KGAT_OK;
    dim3 grid((n + 63) / 64, (m + 63) / 64);
    sgemm_nt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A, lda, B, ldb, C, ldc, m, n, k);
    return check_launch();
}

int kgat_mask_scores(float* scores, int64_t ld, int32_t m, int32_t n, const int32_t* mask_ptr, const int32_t* mask_items, void* stream) {
    if (m < 0 || n < 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (m == 0) return KGAT_OK;
    mask_scores_kernel<<<m, 128, 0, (cudaStream_t)stream>>>(scores, ld, m, n, mask_ptr, mask_items);
    return check_launch();
}

int kgat_topk_rows(const float* scores, int64_t ld, int32_t m, int32_t n, int32_t k, int32_t* idx_out, float* val_out, void* stream) {
    if (m < 0 || n <= 0 || k <= 0 || k > kTopkMax || k > n) return KGAT_ERR_INVALID_ARGUMENT;
    if (m == 0) return KGAT_OK;
    topk_rows_kernel<<<m, kTopkThreads, 0, (cudaStream_t)stream>>>(scores, ld, m, n, k, idx_out, val_out);
    return check_launch();
}

}  // extern "C"
