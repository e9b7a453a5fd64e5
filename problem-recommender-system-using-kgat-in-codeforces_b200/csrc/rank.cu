// Exact full ranking of held-out targets for any number of users without materialising the score matrix (DESIGN section 4.8).
//
// Score s(u, c) = the sequential fmaf chain over the concatenated row E0|E1|...|EL of user u and candidate c (zero-padded to a
// multiple of 16 columns), bit-identical to PREDICT / recommend_topk / recommend.  Key K(u, c) = (float_key(s) << 32) |
// (0xFFFFFFFF - pos(c)), pos = position in the candidate list: exactly recommend's order (topk_rows key descending, then
// earlier position).  For an eligible target p (a candidate not excluded for u):
//
//     rank(u, p) = #{ c eligible for u : K(u, c) > K(u, p) }
//
// so rank < k <= 128 means that recommend(u, items, k, exclude) lists p at position rank.  Only integers are counted, so the
// result does not depend on how the work is split.
//
//   rank_keys_kernel   one warp per user: scores its targets, keeps the eligible ones and sorts their keys ascending by rank
//       selection (keys are unique within a user);
//   rank_count_kernel  one CTA per (64-user tile, candidate slice), recommend_score_kernel's tiles: a score matters only if its
//       key beats the user's lowest target key; then j = #target keys below it (binary search), and if the candidate is not
//       excluded, bucket j - 1 gains one.  The tile's keys and buckets sit in shared memory when they fit (else in global);
//   rank_finalize_kernel  one warp per user: rank of sorted target i = sum of buckets i.., scattered back to item order; the
//       number of eligible candidates.
#include "common.cuh"

namespace kgat {
namespace {

constexpr int kRankSmemTargets = 4096;  // target keys + buckets of one user tile held in shared memory (12 B each)

inline int64_t align256(int64_t b) { return (b + 255) & ~int64_t(255); }

inline int64_t workspace_bytes(int64_t n_users, int64_t n_targets) {
    return align256(n_targets * 8) + 2 * align256(n_targets * 4) + align256(n_users * 4);
}

inline size_t count_smem_bytes(int width_pad) {
    return sizeof(float) * tile_smem_floats(width_pad) + (sizeof(uint64_t) + sizeof(int32_t)) * (size_t)kRankSmemTargets;
}

struct RankArgs {
    ConcatTables T;
    int width_pad;
    const int32_t* users;       // [n_users] table rows
    int n_users;
    const int32_t* cand;        // [n_cand] candidate table rows; position = index
    int n_cand;
    const int32_t* pos_map;     // nullable (then cand[c] == c): position of item x, -1 when not a candidate
    int n_pos;
    const int32_t* tgt_ptr;     // targets of table row u: tgt_items[tgt_ptr[u] .. tgt_ptr[u+1]), ascending
    const int32_t* tgt_items;
    const int64_t* out_ptr;     // [n_users + 1]: row b of the outputs
    const int32_t* excl_ptr;    // nullable
    const int32_t* excl_items;
    int slices;
    uint64_t* skey;             // ws [n_targets]: row b's eligible target keys, ascending, from out_ptr[b]
    int32_t* sidx;              // ws [n_targets]: their index within the row
    int32_t* bucket;            // ws [n_targets]: candidates between sorted keys i and i + 1 (flags while sorting)
    int32_t* n_el;              // ws [n_users]: eligible targets per row
    int64_t* out_items;
    float* out_scores;
    int64_t* out_rank;          // also the unsorted keys while sorting
    int64_t* out_eligible;
};

__device__ __forceinline__ int item_pos(const RankArgs& a, int item) {
    if (!a.pos_map) return item < a.n_cand ? item : -1;
    return item < a.n_pos ? a.pos_map[item] : -1;
}

__device__ __forceinline__ bool in_sorted(const int32_t* p, int n, int x) {
    const int i = lower_bound_i32(p, n, x);
    return i < n && __ldg(p + i) == x;
}

__device__ __forceinline__ uint64_t rank_key(float s, int pos) { return ((uint64_t)float_key(s) << 32) | (0xFFFFFFFFu - (uint32_t)pos); }

// number of entries of the ascending p[0, n) below x
__device__ __forceinline__ int count_below(const uint64_t* p, int n, uint64_t x) {
    int lo = 0;
    while (n > 0) {
        const int half = n >> 1;
        if (p[lo + half] < x) {
            lo += half + 1;
            n -= half + 1;
        } else {
            n = half;
        }
    }
    return lo;
}

// One warp per user row b.
__global__ void __launch_bounds__(256) rank_keys_kernel(RankArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (b >= a.n_users) return;
    const int u = a.users[b];
    const int64_t o = a.out_ptr[b];
    const int n_t = (int)(a.out_ptr[b + 1] - o);
    const int32_t* tl = a.tgt_items + a.tgt_ptr[u];
    int eb = 0, en = 0;
    if (a.excl_ptr) {
        eb = a.excl_ptr[u];
        en = a.excl_ptr[u + 1] - eb;
    }
    const int nq = a.width_pad / 4;
    uint64_t* key = reinterpret_cast<uint64_t*>(a.out_rank + o);
    int32_t* flag = a.bucket + o;
    int n_elig = 0;
    for (int t = lane; t < n_t; t += 32) {
        const int item = tl[t];
        float s = 0.f;
        for (int q = 0; q < nq; ++q) {
            const float4 x = concat_quad(a.T, u, q), y = concat_quad(a.T, item, q);
            s = fmaf(x.x, y.x, s);
            s = fmaf(x.y, y.y, s);
            s = fmaf(x.z, y.z, s);
            s = fmaf(x.w, y.w, s);
        }
        a.out_items[o + t] = item;
        a.out_scores[o + t] = s;
        const int pos = item_pos(a, item);
        const bool elig = pos >= 0 && !(en > 0 && in_sorted(a.excl_items + eb, en, item));
        key[t] = elig ? rank_key(s, pos) : 0;
        flag[t] = elig;
        n_elig += elig;
    }
    __syncwarp();
    // rank selection: keys are unique within the row, so the eligible keys below mine give my sorted index
    for (int t = lane; t < n_t; t += 32) {
        if (!flag[t]) continue;
        const uint64_t k = key[t];
        int r = 0;
        for (int v = 0; v < n_t; ++v) r += flag[v] && key[v] < k;
        a.skey[o + r] = k;
        a.sidx[o + r] = t;
    }
    __syncwarp();
    for (int t = lane; t < n_t; t += 32) {
        a.out_rank[o + t] = -1;  // eligible targets get their rank in rank_finalize_kernel
        flag[t] = 0;             // the buckets start at zero
    }
    n_elig = __reduce_add_sync(kFull, n_elig);
    if (lane == 0) a.n_el[b] = n_elig;
}

__global__ void __launch_bounds__(kTileThreads) rank_count_kernel(RankArgs a) {
    extern __shared__ float4 smem_f4[];
    float* Us = reinterpret_cast<float*>(smem_f4);                        // [width_pad][kTilePad]: the tile's users, transposed
    float* Bs = Us + (size_t)a.width_pad * kTilePad;                      // [16][kTilePad]: one 16-column slab of a candidate tile
    uint64_t* s_key = reinterpret_cast<uint64_t*>(Bs + 16 * kTilePad);    // [kRankSmemTargets]
    int32_t* s_bucket = reinterpret_cast<int32_t*>(s_key + kRankSmemTargets);

    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const int u0 = blockIdx.x * kTileUsers;
    const int u_end = min(u0 + kTileUsers, a.n_users);
    const int c_begin = (int)((int64_t)a.n_cand * blockIdx.y / a.slices), c_end = (int)((int64_t)a.n_cand * (blockIdx.y + 1) / a.slices);
    const int64_t t0 = a.out_ptr[u0];
    const int64_t t_n = a.out_ptr[u_end] - t0;
    // the tile's sorted keys and buckets: shared memory when they fit, else the workspace itself
    const bool local = t_n <= kRankSmemTargets;
    const uint64_t* keys = local ? s_key : a.skey + t0;
    int32_t* buckets = local ? s_bucket : a.bucket + t0;

    stage_user_tile(a.T, a.users, a.n_users, u0, a.width_pad, Us);
    if (local) {
        for (int e = tid; e < t_n; e += kTileThreads) {
            s_key[e] = a.skey[t0 + e];
            s_bucket[e] = 0;
        }
    }
    // per-thread: its 4 users' key ranges, lowest key and exclusion ranges
    int kb[4], kn[4], ex_b[4], ex_n[4];
    uint64_t kmin[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int u = u0 + ty * 4 + i;
        kb[i] = kn[i] = ex_b[i] = ex_n[i] = 0;
        kmin[i] = 0;
        if (u < a.n_users) {
            kb[i] = (int)(a.out_ptr[u] - t0);
            kn[i] = a.n_el[u];
            if (kn[i] > 0) kmin[i] = a.skey[t0 + kb[i]];
            if (a.excl_ptr) {
                const int id = a.users[u];
                ex_b[i] = a.excl_ptr[id];
                ex_n[i] = a.excl_ptr[id + 1] - ex_b[i];
            }
        }
    }
    __syncthreads();

    for (int c0 = c_begin; c0 < c_end; c0 += kTileItems) {
        float acc[4][4];
        score_tile(a.T, a.cand, c0, c_end, a.width_pad, Us, Bs, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (kn[i] == 0) continue;
            int run_b = -1, run_n = 0;  // consecutive hits of one bucket go in one atomic
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + tx * 4 + j;
                if (c >= c_end) continue;
                const uint64_t K = rank_key(acc[i][j], c);
                if (K <= kmin[i]) continue;
                const int bj = count_below(keys + kb[i], kn[i], K) - 1;
                if (ex_n[i] > 0 && in_sorted(a.excl_items + ex_b[i], ex_n[i], a.cand[c])) continue;
                if (bj != run_b) {
                    if (run_n) atomicAdd(buckets + kb[i] + run_b, run_n);
                    run_b = bj;
                    run_n = 0;
                }
                ++run_n;
            }
            if (run_n) atomicAdd(buckets + kb[i] + run_b, run_n);
        }
    }
    if (local) {
        __syncthreads();
        for (int e = tid; e < t_n; e += kTileThreads) {
            const int v = s_bucket[e];
            if (v) atomicAdd(a.bucket + t0 + e, v);
        }
    }
}

// One warp per user row b: suffix sums of the buckets from the top, scattered to item order; eligible candidates.
__global__ void __launch_bounds__(256) rank_finalize_kernel(RankArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (b >= a.n_users) return;
    const int64_t o = a.out_ptr[b];
    const int P = a.n_el[b];
    int64_t carry = 0;
    for (int base = ((P + 31) / 32 - 1) * 32; base >= 0; base -= 32) {
        const int r = base + lane;
        int64_t v = r < P ? a.bucket[o + r] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t w = __shfl_down_sync(kFull, v, d);
            if (lane + d < 32) v += w;
        }
        if (r < P) a.out_rank[o + a.sidx[o + r]] = carry + v;
        carry += __shfl_sync(kFull, v, 0);
    }
    int n_ex = 0;
    if (a.excl_ptr) {
        const int u = a.users[b];
        for (int e = a.excl_ptr[u] + lane; e < a.excl_ptr[u + 1]; e += 32) n_ex += item_pos(a, a.excl_items[e]) >= 0;
    }
    n_ex = __reduce_add_sync(kFull, n_ex);
    if (lane == 0) a.out_eligible[b] = a.n_cand - n_ex;
}

// Dynamic shared memory of the count kernel at this width (opted in on the current device) and how many of its CTAs fit on
// one SM.  KGAT_ERR_UNSUPPORTED when one CTA does not fit.
int count_plan(const ConcatTables& T, size_t* smem, int* per_sm) {
    *smem = count_smem_bytes(padded_width(T));
    int dev = 0, max_smem = 0;
    KGAT_CUDA_TRY(cudaGetDevice(&dev));
    KGAT_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (*smem > (size_t)max_smem) return KGAT_ERR_UNSUPPORTED;
    KGAT_CUDA_TRY(cudaFuncSetAttribute(rank_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem));
    KGAT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, rank_count_kernel, kTileThreads, *smem));
    if (*per_sm < 1) *per_sm = 1;
    return KGAT_OK;
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int64_t kgat_rank_workspace_bytes(const kgat_tables_t* tables, int64_t n_users, int64_t n_targets) {
    ConcatTables T;
    if (!tables_from(tables, &T) || n_users < 0 || n_targets < 0) return -1;
    size_t smem = 0;
    int per_sm = 1;
    if (count_plan(T, &smem, &per_sm) != KGAT_OK) return -1;
    return workspace_bytes(n_users, n_targets);
}

int kgat_rank_targets(const kgat_tables_t* tables, const int32_t* users, int64_t n_users, const int32_t* cand_items, int64_t n_cand,
                      const int32_t* pos_map, int64_t n_pos, const int32_t* target_ptr, const int32_t* target_items, const int64_t* out_ptr,
                      int64_t n_targets, const int32_t* exclude_ptr, const int32_t* exclude_items, int32_t slices, int64_t* out_items,
                      float* out_scores, int64_t* out_rank, int64_t* out_eligible, void* workspace, int64_t workspace_bytes_, void* stream) {
    ConcatTables T;
    if (!tables_from(tables, &T) || n_users < 0 || n_users > 0x7fffffff || n_cand < 0 || n_cand > 0x7fffffff || n_pos < 0 || n_pos > 0x7fffffff ||
        n_targets < 0 || slices < 0 || slices > kTileMaxSlices)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (n_users == 0) return KGAT_OK;
    if (!users || (n_cand > 0 && !cand_items) || (pos_map && n_pos == 0) || !target_ptr || (n_targets > 0 && !target_items) || !out_ptr ||
        (exclude_ptr && !exclude_items) || !out_eligible || (n_targets > 0 && (!out_items || !out_scores || !out_rank)) || !workspace)
        return KGAT_ERR_INVALID_ARGUMENT;
    size_t smem = 0;
    int per_sm = 1;
    const int rc_plan = count_plan(T, &smem, &per_sm);
    if (rc_plan != KGAT_OK) return rc_plan;
    if (workspace_bytes_ < workspace_bytes(n_users, n_targets)) return KGAT_ERR_WORKSPACE;
    RankArgs a;
    a.T = T;
    a.width_pad = padded_width(T);
    a.users = users;
    a.n_users = (int)n_users;
    a.cand = cand_items;
    a.n_cand = (int)n_cand;
    a.pos_map = pos_map;
    a.n_pos = (int)n_pos;
    a.tgt_ptr = target_ptr;
    a.tgt_items = target_items;
    a.out_ptr = out_ptr;
    a.excl_ptr = exclude_ptr;
    a.excl_items = exclude_items;
    a.slices = pick_slices(n_users, n_cand, per_sm, slices);
    char* w = static_cast<char*>(workspace);
    a.skey = reinterpret_cast<uint64_t*>(w);
    w += align256(n_targets * 8);
    a.sidx = reinterpret_cast<int32_t*>(w);
    w += align256(n_targets * 4);
    a.bucket = reinterpret_cast<int32_t*>(w);
    w += align256(n_targets * 4);
    a.n_el = reinterpret_cast<int32_t*>(w);
    a.out_items = out_items;
    a.out_scores = out_scores;
    a.out_rank = out_rank;
    a.out_eligible = out_eligible;
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned warp_blocks = (unsigned)((n_users * 32 + 255) / 256);
    rank_keys_kernel<<<warp_blocks, 256, 0, s>>>(a);
    int rc = check_launch();
    if (rc != KGAT_OK) return rc;
    if (n_cand > 0 && n_targets > 0) {
        const dim3 grid((unsigned)((n_users + kTileUsers - 1) / kTileUsers), (unsigned)a.slices);
        rank_count_kernel<<<grid, kTileThreads, smem, s>>>(a);
        rc = check_launch();
        if (rc != KGAT_OK) return rc;
    }
    rank_finalize_kernel<<<warp_blocks, 256, 0, s>>>(a);
    return check_launch();
}

}  // extern "C"
