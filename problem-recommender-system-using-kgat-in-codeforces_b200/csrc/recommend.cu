// Filtered top-k recommendations for any number of users without materialising the score matrix (DESIGN section 4.7).
//
// Score s(u, c) = the sequential fmaf chain over the concatenated row E0|E1|...|EL of user u and candidate c, in ascending
// column order from +0, padded with zero columns to a multiple of 16 -- the arithmetic of sgemm_nt_kernel, so every score is
// bit-identical to PREDICT / recommend_topk.  Order: descending float_key(score) (the topk_rows key), then ascending
// candidate index; candidate indices ascend with the position in the caller's item list, so this is the documented order.
// It is total, so the result does not depend on how the candidates are split over CTAs.
//
//   recommend_flag_kernel / recommend_compact_kernel  (only with a filter)  keep the items whose CKG node has a stored
//       entry towards one entity of every group, in input order;
//   recommend_score_kernel  one CTA per (64-user tile, candidate slice): the tile's concatenated user rows stay in shared
//       memory, the slice is walked in 64-candidate tiles with the sgemm_nt 4 x 4 micro-tile, and every user keeps a
//       running top-k (a score enters a pending buffer only when it beats the user's current k-th entry and is not
//       excluded; the buffer is folded into the top-k by rank selection after each tile);
//   recommend_merge_kernel  one warp per user merges the slices' sorted lists by rank and writes the padded outputs.
#include "common.cuh"

namespace kgat {
namespace {

constexpr int kRecThreads = kTileThreads;
constexpr int kRecUsers = kTileUsers;  // users per CTA
constexpr int kRecItems = kTileItems;  // candidates per tile
constexpr int kRecMaxK = kTopkMaxK;
constexpr int kRecMaxSlices = kTileMaxSlices;

inline int64_t align256(int64_t b) { return (b + 255) & ~int64_t(255); }

inline int64_t workspace_bytes(int64_t n_users, int slices, int k) {
    return align256(n_users * slices * k * (int64_t)sizeof(Entry)) + align256(n_users * slices * 4);
}

inline size_t score_smem_bytes(int width_pad, int k) {
    return sizeof(float) * tile_smem_floats(width_pad) + sizeof(Entry) * (size_t)kRecUsers * (k + kRecItems) + 2 * sizeof(int) * kRecUsers;
}

// ---------------------------------------------------------------------------------------------------------------------
// filter
// ---------------------------------------------------------------------------------------------------------------------
// One warp per item: flag[i] = 1 iff row (user_num + items[i]) of A has a column in every group of entity nodes.
__global__ void __launch_bounds__(256) recommend_flag_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col_idx,
                                                             int user_num, const int32_t* __restrict__ items, int n_items,
                                                             const int32_t* __restrict__ group_ptr, const int32_t* __restrict__ group_nodes,
                                                             int n_groups, int32_t* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (i >= n_items) return;
    const int node = user_num + items[i];
    const int rb = row_ptr[node], deg = row_ptr[node + 1] - rb;
    bool pass = true;
    for (int g = 0; g < n_groups && pass; ++g) {
        bool hit = false;
        for (int e = group_ptr[g] + lane; e < group_ptr[g + 1] && !hit; e += 32) {
            const int x = group_nodes[e];
            const int p = lower_bound_i32(col_idx + rb, deg, x);
            hit = p < deg && col_idx[rb + p] == x;
        }
        pass = __any_sync(kFull, hit);
    }
    if (lane == 0) flag[i] = pass ? 1 : 0;
}

// One CTA, in place: pos[0, n) holds the flags on entry and the passing positions (ascending) on exit; cand[j] = items[pos[j]],
// *n_cand = their number.
__global__ void __launch_bounds__(1024) recommend_compact_kernel(const int32_t* __restrict__ items, int n_items, int32_t* __restrict__ pos,
                                                                 int32_t* __restrict__ cand, int32_t* __restrict__ n_cand) {
    __shared__ int warp_tot[32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int b = 0; b < n_items; b += 1024) {
        const int i = b + tid;
        const bool keep = i < n_items && pos[i] != 0;
        const unsigned bal = __ballot_sync(kFull, keep);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();  // every flag of this chunk is read before any position of it is written
        int before = s_base + __popc(bal & ((1u << lane) - 1));
        int tot = 0;
        for (int w = 0; w < 32; ++w) {
            if (w < warp) before += warp_tot[w];
            tot += warp_tot[w];
        }
        if (keep) {
            pos[before] = i;
            cand[before] = items[i];
        }
        __syncthreads();
        if (tid == 0) s_base += tot;
        __syncthreads();
    }
    if (tid == 0) *n_cand = s_base;
}

// ---------------------------------------------------------------------------------------------------------------------
// fused score + running top-k
// ---------------------------------------------------------------------------------------------------------------------
struct ScoreArgs {
    ConcatTables T;
    int width_pad;
    const int32_t* users;
    int n_users;
    const int32_t* cand;
    int n_cand_max;
    const int32_t* n_cand_dev;  // nullable: n_cand_max candidates
    int k;
    const int32_t* excl_ptr;    // nullable
    const int32_t* excl_items;
    int slices;
    Entry* ws_list;             // [n_users][slices][k]
    int32_t* ws_len;            // [n_users][slices]
};

__global__ void __launch_bounds__(kRecThreads) recommend_score_kernel(ScoreArgs a) {
    extern __shared__ float4 smem_f4[];
    float* Us = reinterpret_cast<float*>(smem_f4);              // [width_pad][kTilePad]: the tile's users, transposed
    float* Bs = Us + (size_t)a.width_pad * kTilePad;            // [16][kTilePad]: one 16-column slab of a candidate tile
    Entry* top = reinterpret_cast<Entry*>(Bs + 16 * kTilePad);  // [kRecUsers][k], sorted best-first
    Entry* pend = top + kRecUsers * a.k;                        // [kRecUsers][kRecItems], unordered
    int* n_top = reinterpret_cast<int*>(pend + kRecUsers * kRecItems);
    int* n_pend = n_top + kRecUsers;

    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16, lane = tid & 31, warp = tid >> 5;
    const int u0 = blockIdx.x * kRecUsers;
    const int slice = blockIdx.y;
    const int k = a.k;
    const int n_cand = a.n_cand_dev ? *a.n_cand_dev : a.n_cand_max;
    const int c_begin = (int)((int64_t)n_cand * slice / a.slices), c_end = (int)((int64_t)n_cand * (slice + 1) / a.slices);

    // stage the users' concatenated rows (zero rows past n_users, zero columns past the width)
    stage_user_tile(a.T, a.users, a.n_users, u0, a.width_pad, Us);
    if (tid < kRecUsers) { n_top[tid] = 0; n_pend[tid] = 0; }

    // per-thread exclusion ranges of its 4 users
    int ex_b[4], ex_n[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int u = u0 + ty * 4 + i;
        ex_b[i] = ex_n[i] = 0;
        if (a.excl_ptr && u < a.n_users) {
            const int id = a.users[u];
            ex_b[i] = a.excl_ptr[id];
            ex_n[i] = a.excl_ptr[id + 1] - ex_b[i];
        }
    }
    __syncthreads();

    for (int c0 = c_begin; c0 < c_end; c0 += kRecItems) {
        float acc[4][4];
        score_tile(a.T, a.cand, c0, c_end, a.width_pad, Us, Bs, acc);
        // admission: beats the user's k-th entry (or the list is not full) and is not excluded
        bool any = false;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int ul = ty * 4 + i;
            if (u0 + ul >= a.n_users) continue;
            const int nt = n_top[ul];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const Entry x{acc[i][j], c0 + tx * 4 + j};
                if (x.c >= c_end) continue;
                if (nt == k && !beats(x, top[ul * k + k - 1])) continue;
                if (ex_n[i] > 0) {
                    const int item = a.cand[x.c];
                    const int p = lower_bound_i32(a.excl_items + ex_b[i], ex_n[i], item);
                    if (p < ex_n[i] && a.excl_items[ex_b[i] + p] == item) continue;
                }
                pend[ul * kRecItems + atomicAdd(&n_pend[ul], 1)] = x;
                any = true;
            }
        }
        if (!__syncthreads_or(any)) continue;
        // fold each user's pending entries into its top-k: rank = members of the union that beat it (a total order)
        for (int ul = warp; ul < kRecUsers; ul += kRecThreads / 32) {
            const int np = n_pend[ul];
            if (np == 0) continue;
            const int n_new = fold_pending(top + ul * k, n_top[ul], pend + ul * kRecItems, np, k, lane);
            if (lane == 0) {
                n_top[ul] = n_new;
                n_pend[ul] = 0;
            }
            __syncwarp();
        }
        __syncthreads();
    }
    for (int ul = warp; ul < kRecUsers; ul += kRecThreads / 32) {
        const int u = u0 + ul;
        if (u >= a.n_users) break;
        const int nt = n_top[ul];
        const int64_t o = (int64_t)u * a.slices + slice;
        for (int i = lane; i < nt; i += 32) a.ws_list[o * k + i] = top[ul * k + i];
        if (lane == 0) a.ws_len[o] = nt;
    }
}

// One warp per user: rank of a slice's entry = its index + the entries of the other slices that beat it.
__global__ void __launch_bounds__(256) recommend_merge_kernel(const Entry* __restrict__ ws_list, const int32_t* __restrict__ ws_len, int n_users,
                                                              int slices, int k, const int32_t* __restrict__ cand, int64_t* __restrict__ out_items,
                                                              float* __restrict__ out_scores, int32_t* __restrict__ out_count) {
    const int lane = threadIdx.x & 31;
    const int64_t u = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (u >= n_users) return;
    const int total = merge_slices(ws_list + u * slices * k, ws_len + u * slices, slices, k, lane, [&](int r, const Entry& x) {
        out_items[u * k + r] = cand[x.c];
        out_scores[u * k + r] = x.s;
    });
    for (int r = total + lane; r < k; r += 32) {
        out_items[u * k + r] = -1;
        out_scores[u * k + r] = -INFINITY;
    }
    if (lane == 0) out_count[u] = total;
}

// Dynamic shared memory of the score kernel at this width and k (opted in on the current device) and how many of its CTAs
// fit on one SM.  KGAT_ERR_UNSUPPORTED when one CTA does not fit.
int score_plan(const ConcatTables& T, int k, size_t* smem, int* per_sm) {
    *smem = score_smem_bytes(padded_width(T), k);
    int dev = 0, max_smem = 0;
    KGAT_CUDA_TRY(cudaGetDevice(&dev));
    KGAT_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (*smem > (size_t)max_smem) return KGAT_ERR_UNSUPPORTED;
    KGAT_CUDA_TRY(cudaFuncSetAttribute(recommend_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem));
    KGAT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, recommend_score_kernel, kRecThreads, *smem));
    if (*per_sm < 1) *per_sm = 1;
    return KGAT_OK;
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int kgat_recommend_filter(const int32_t* row_ptr, const int32_t* col_idx, int64_t n_nodes, int32_t user_num, const int32_t* items,
                          int64_t n_items, const int32_t* group_ptr, const int32_t* group_nodes, int32_t n_groups, int32_t* positions,
                          int32_t* cand_items, int32_t* n_cand, void* stream) {
    if (n_nodes < 0 || n_nodes > 0x7fffffff || user_num < 0 || n_items < 0 || n_items > 0x7fffffff || n_groups < 0)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (!row_ptr || !col_idx || !group_ptr || !n_cand || (n_groups > 0 && !group_nodes) || (n_items > 0 && (!items || !positions || !cand_items)))
        return KGAT_ERR_INVALID_ARGUMENT;
    cudaStream_t s = (cudaStream_t)stream;
    if (n_items > 0) {
        recommend_flag_kernel<<<(unsigned)((n_items * 32 + 255) / 256), 256, 0, s>>>(row_ptr, col_idx, user_num, items, (int)n_items, group_ptr,
                                                                                    group_nodes, n_groups, positions);
        const int rc = check_launch();
        if (rc != KGAT_OK) return rc;
    }
    recommend_compact_kernel<<<1, 1024, 0, s>>>(items, (int)n_items, positions, cand_items, n_cand);
    return check_launch();
}

int64_t kgat_recommend_workspace_bytes(const kgat_tables_t* tables, int64_t n_users, int64_t n_cand_max, int32_t k, int32_t slices) {
    ConcatTables T;
    if (!tables_from(tables, &T) || n_users < 0 || n_cand_max < 0 || k < 1 || k > kRecMaxK || slices < 0 || slices > kRecMaxSlices) return -1;
    size_t smem = 0;
    int per_sm = 1;
    if (score_plan(T, k, &smem, &per_sm) != KGAT_OK) return -1;
    return workspace_bytes(n_users, pick_slices(n_users, n_cand_max, per_sm, slices), k);
}

int kgat_recommend_topk(const kgat_tables_t* tables, const int32_t* users, int64_t n_users, const int32_t* cand_items, int64_t n_cand_max,
                        const int32_t* n_cand, int32_t k, const int32_t* exclude_ptr, const int32_t* exclude_items, int32_t slices,
                        int64_t* out_items, float* out_scores, int32_t* out_count, void* workspace, int64_t workspace_bytes_, void* stream) {
    ConcatTables T;
    if (!tables_from(tables, &T) || n_users < 0 || n_users > 0x7fffffff || n_cand_max < 0 || n_cand_max > 0x7fffffff || k < 1 || k > kRecMaxK ||
        slices < 0 || slices > kRecMaxSlices)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (n_users == 0) return KGAT_OK;
    if (!users || (n_cand_max > 0 && !cand_items) || (exclude_ptr && !exclude_items) || !out_items || !out_scores || !out_count || !workspace)
        return KGAT_ERR_INVALID_ARGUMENT;
    size_t smem = 0;
    int per_sm = 1;
    const int rc_plan = score_plan(T, k, &smem, &per_sm);
    if (rc_plan != KGAT_OK) return rc_plan;
    const int S = pick_slices(n_users, n_cand_max, per_sm, slices);
    if (workspace_bytes_ < workspace_bytes(n_users, S, k)) return KGAT_ERR_WORKSPACE;
    ScoreArgs a;
    a.T = T;
    a.width_pad = padded_width(T);
    a.users = users;
    a.n_users = (int)n_users;
    a.cand = cand_items;
    a.n_cand_max = (int)n_cand_max;
    a.n_cand_dev = n_cand;
    a.k = k;
    a.excl_ptr = exclude_ptr;
    a.excl_items = exclude_items;
    a.slices = S;
    char* w = static_cast<char*>(workspace);
    a.ws_list = reinterpret_cast<Entry*>(w);
    a.ws_len = reinterpret_cast<int32_t*>(w + align256(n_users * S * k * (int64_t)sizeof(Entry)));
    cudaStream_t s = (cudaStream_t)stream;
    const dim3 grid((unsigned)((n_users + kRecUsers - 1) / kRecUsers), (unsigned)S);
    recommend_score_kernel<<<grid, kRecThreads, smem, s>>>(a);
    int rc = check_launch();
    if (rc != KGAT_OK) return rc;
    recommend_merge_kernel<<<(unsigned)((n_users * 32 + 255) / 256), 256, 0, s>>>(a.ws_list, a.ws_len, (int)n_users, S, k, cand_items, out_items,
                                                                                 out_scores, out_count);
    return check_launch();
}

}  // extern "C"
