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
//
// Capped top-k (DESIGN section 4.10) runs in rounds over the rows still active:
//   recommend_mask_kernel  the groups of each candidate as a 128-bit mask (the filter's membership test);
//   recommend_score_kernel<true>  the score kernel's top-m, admitting only entries after the row's bound (its last entry of
//       the previous round) that touch none of its saturated groups; skipping them is exact, since counts only grow;
//   recommend_capped_greedy_kernel  one warp per row merges the slices, walks the merged list, accepts entries whose groups
//       are all below their caps, and passes the unfinished rows on to the next round.
#include "common.cuh"

namespace kgat {
namespace {

constexpr int kRecThreads = kTileThreads;
constexpr int kRecUsers = kTileUsers;  // users per CTA
constexpr int kRecItems = kTileItems;  // candidates per tile
constexpr int kRecMaxK = kTopkMaxK;
constexpr int kRecMaxSlices = kTileMaxSlices;
constexpr int kCapMaxGroups = 128;  // bits of a candidate's group mask

inline int64_t align256(int64_t b) { return (b + 255) & ~int64_t(255); }

inline int64_t workspace_bytes(int64_t n_users, int slices, int k) {
    return align256(n_users * slices * k * (int64_t)sizeof(Entry)) + align256(n_users * slices * 4);
}

inline size_t score_smem_bytes(int width_pad, int k, bool capped) {
    return sizeof(float) * tile_smem_floats(width_pad) + sizeof(Entry) * (size_t)kRecUsers * (k + kRecItems) + 2 * sizeof(int) * kRecUsers +
           (capped ? (sizeof(uint64_t) + sizeof(uint4)) * kRecUsers : 0);
}

// ---------------------------------------------------------------------------------------------------------------------
// filter
// ---------------------------------------------------------------------------------------------------------------------
// Whole warp: true iff the sorted CSR row col_idx[rb, rb + deg) has a column among group g's entity nodes.
__device__ __forceinline__ bool group_hit(const int32_t* __restrict__ col_idx, int rb, int deg, const int32_t* __restrict__ group_ptr,
                                          const int32_t* __restrict__ group_nodes, int g, int lane) {
    bool hit = false;
    for (int e = group_ptr[g] + lane; e < group_ptr[g + 1] && !hit; e += 32) {
        const int x = group_nodes[e];
        const int p = lower_bound_i32(col_idx + rb, deg, x);
        hit = p < deg && col_idx[rb + p] == x;
    }
    return __any_sync(kFull, hit);
}

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
    for (int g = 0; g < n_groups && pass; ++g) pass = group_hit(col_idx, rb, deg, group_ptr, group_nodes, g, lane);
    if (lane == 0) flag[i] = pass ? 1 : 0;
}

// One warp per candidate position c < n (n = *n_cand when given): bit g of mask[c] (word g / 32, bit g % 32) = row
// (user_num + cand[c]) of A has a column in group g.  n_groups <= kCapMaxGroups.
__global__ void __launch_bounds__(256) recommend_mask_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col_idx,
                                                             int user_num, const int32_t* __restrict__ cand, int n_cand_max,
                                                             const int32_t* __restrict__ n_cand_dev, const int32_t* __restrict__ group_ptr,
                                                             const int32_t* __restrict__ group_nodes, int n_groups, uint4* __restrict__ mask) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (i >= (n_cand_dev ? *n_cand_dev : n_cand_max)) return;
    const int node = user_num + cand[i];
    const int rb = row_ptr[node], deg = row_ptr[node + 1] - rb;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int q = 0; q < 4; ++q)
        for (int g = 32 * q; g < n_groups && g < 32 * q + 32; ++g)
            if (group_hit(col_idx, rb, deg, group_ptr, group_nodes, g, lane)) w[q] |= 1u << (g & 31);
    if (lane == 0) mask[i] = make_uint4(w[0], w[1], w[2], w[3]);
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

// Row state of a capped round (kgat_recommend_capped_round): the score kernel admits an entry only when it comes after the
// row's bound and its group mask misses the row's saturated groups.  Staged user u is row rows[u] (u itself in the first
// round, rows == nullptr, when no row has a bound yet and the saturated groups are those with cap 0).
struct CapArgs {
    const int32_t* rows;   // nullable
    const Entry* bound;    // [n_rows]: the last entry of the row's previous round
    const uint4* sat;      // [n_rows]: saturated groups
    const uint4* mask;     // [n_cand]: groups of each candidate
    const int32_t* caps;   // [n_groups]
    int n_groups;
};

// beats as one integer: a beats b iff entry_key(a) > entry_key(b); every key is below ~0, the key of "no bound"
__device__ __forceinline__ uint64_t entry_key(const Entry& x) { return ((uint64_t)float_key(x.s) << 32) | (uint32_t)(0x7fffffff - x.c); }

template <bool kCapped> struct ScoreParams : ScoreArgs {};
template <> struct ScoreParams<true> : ScoreArgs { CapArgs cap; };

template <bool kCapped>
__global__ void __launch_bounds__(kRecThreads) recommend_score_kernel(ScoreParams<kCapped> a) {
    extern __shared__ float4 smem_f4[];
    float* Us = reinterpret_cast<float*>(smem_f4);              // [width_pad][kTilePad]: the tile's users, transposed
    float* Bs = Us + (size_t)a.width_pad * kTilePad;            // [16][kTilePad]: one 16-column slab of a candidate tile
    Entry* top = reinterpret_cast<Entry*>(Bs + 16 * kTilePad);  // [kRecUsers][k], sorted best-first
    Entry* pend = top + kRecUsers * a.k;                        // [kRecUsers][kRecItems], unordered
    int* n_top = reinterpret_cast<int*>(pend + kRecUsers * kRecItems);
    int* n_pend = n_top + kRecUsers;
    uint64_t* s_bkey = reinterpret_cast<uint64_t*>(n_pend + kRecUsers);  // capped: [kRecUsers]
    uint4* s_sat = reinterpret_cast<uint4*>(s_bkey + kRecUsers);        // capped: [kRecUsers]

    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16, lane = tid & 31, warp = tid >> 5;
    const int u0 = blockIdx.x * kRecUsers;
    const int slice = blockIdx.y;
    const int k = a.k;
    const int n_cand = a.n_cand_dev ? *a.n_cand_dev : a.n_cand_max;
    const int c_begin = (int)((int64_t)n_cand * slice / a.slices), c_end = (int)((int64_t)n_cand * (slice + 1) / a.slices);

    // stage the users' concatenated rows (zero rows past n_users, zero columns past the width)
    stage_user_tile(a.T, a.users, a.n_users, u0, a.width_pad, Us);
    if (tid < kRecUsers) { n_top[tid] = 0; n_pend[tid] = 0; }
    if constexpr (kCapped) {
        if (tid < kRecUsers) {
            uint64_t bkey = ~0ull;
            uint4 sat = make_uint4(0u, 0u, 0u, 0u);
            if (!a.cap.rows) {
                for (int g = 0; g < a.cap.n_groups; ++g) {
                    const uint32_t bit = a.cap.caps[g] == 0 ? 1u << (g & 31) : 0u;
                    if (g < 32) sat.x |= bit; else if (g < 64) sat.y |= bit; else if (g < 96) sat.z |= bit; else sat.w |= bit;
                }
            } else if (u0 + tid < a.n_users) {
                const int row = a.cap.rows[u0 + tid];
                bkey = entry_key(a.cap.bound[row]);
                sat = a.cap.sat[row];
            }
            s_bkey[tid] = bkey;
            s_sat[tid] = sat;
        }
    }

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
        // admission: beats the user's k-th entry (or the list is not full) and is not excluded; capped: comes after the
        // row's bound and touches none of its saturated groups
        bool any = false;
        uint4 cm[4];  // capped: the group masks of the thread's 4 candidates
        if constexpr (kCapped) {
#pragma unroll
            for (int j = 0; j < 4; ++j) cm[j] = c0 + tx * 4 + j < c_end ? a.cap.mask[c0 + tx * 4 + j] : make_uint4(0u, 0u, 0u, 0u);
        }
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
                if constexpr (kCapped) {
                    if (entry_key(x) >= s_bkey[ul]) continue;
                    const uint4 sat = s_sat[ul];
                    if ((cm[j].x & sat.x) | (cm[j].y & sat.y) | (cm[j].z & sat.z) | (cm[j].w & sat.w)) continue;
                }
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

// One warp per active row of a capped round: merges the slices' lists into shared memory, walks them in order, accepts an
// entry when none of its groups is at its cap, appends it to the row's output and counts it in each of its groups.  The row
// is finished at k acceptances or when the round found fewer than m entries; then its padding is written.  Otherwise its
// counts, saturated groups and bound (the round's last entry) are stored and it is appended to the next round's list.
struct GreedyArgs {
    const Entry* ws_list;    // [n_active][slices][m]
    const int32_t* ws_len;   // [n_active][slices]
    int slices, m, k, n_active, n_groups;
    const int32_t* rows_in;  // nullable (first round): active slot j is row j
    const int32_t* users;    // [n_rows]
    const int32_t* cand;
    const uint4* mask;
    const int32_t* caps;
    uint8_t* counts;         // [n_rows][n_groups]
    Entry* bound;            // [n_rows]
    uint4* sat;              // [n_rows]
    int32_t* rows_out;       // next round: rows and their users, *n_out of them
    int32_t* users_out;
    int32_t* n_out;
    int64_t* out_items;
    float* out_scores;
    int32_t* out_count;
};

__global__ void __launch_bounds__(256) recommend_capped_greedy_kernel(GreedyArgs a) {
    __shared__ Entry s_list[256 / 32][kRecMaxK];
    const int lane = threadIdx.x & 31;
    const int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (j >= a.n_active) return;
    const bool first = a.rows_in == nullptr;
    const int row = first ? (int)j : a.rows_in[j];
    const int m = a.m, k = a.k, G = a.n_groups;
    Entry* l = s_list[threadIdx.x >> 5];
    const int total = merge_slices(a.ws_list + j * a.slices * m, a.ws_len + j * a.slices, a.slices, m, lane, [&](int r, const Entry& x) { l[r] = x; });
    __syncwarp();
    // lane owns groups lane + 32 q
    int cnt[4], cap[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int g = 32 * q + lane;
        cap[q] = g < G ? a.caps[g] : 0x7fffffff;
        cnt[q] = !first && g < G ? a.counts[(int64_t)row * G + g] : 0;
    }
    int n = first ? 0 : a.out_count[row];
    int64_t* oi = a.out_items + (int64_t)row * k;
    float* os = a.out_scores + (int64_t)row * k;
    for (int i = 0; i < total && n < k; ++i) {
        const Entry x = l[i];
        const uint4 mk = a.mask[x.c];
        const uint32_t w[4] = {mk.x, mk.y, mk.z, mk.w};
        bool full = false;
#pragma unroll
        for (int q = 0; q < 4; ++q) full |= ((w[q] >> lane) & 1u) && cnt[q] >= cap[q];
        if (__any_sync(kFull, full)) continue;
#pragma unroll
        for (int q = 0; q < 4; ++q) cnt[q] += (w[q] >> lane) & 1u;
        if (lane == 0) {
            oi[n] = a.cand[x.c];
            os[n] = x.s;
        }
        ++n;
    }
    if (n == k || total < m) {
        for (int r = n + lane; r < k; r += 32) {
            oi[r] = -1;
            os[r] = -INFINITY;
        }
    } else {
        uint32_t sat[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int g = 32 * q + lane;
            if (g < G) a.counts[(int64_t)row * G + g] = (uint8_t)cnt[q];
            sat[q] = __ballot_sync(kFull, cnt[q] >= cap[q]);
        }
        if (lane == 0) {
            a.sat[row] = make_uint4(sat[0], sat[1], sat[2], sat[3]);
            a.bound[row] = l[m - 1];
            const int slot = atomicAdd(a.n_out, 1);  // the slot order does not change any row's result
            a.rows_out[slot] = row;
            a.users_out[slot] = a.users[row];
        }
    }
    if (lane == 0) a.out_count[row] = n;
}

// Workspace of a capped call over n_rows rows: the score lists of up to `slots` (active row, slice) pairs, then the row state
// and the two active lists (rows, users) that alternate between rounds.
struct CapLayout {
    int64_t len, counts, bound, sat, rows[2], users[2], total;
};

inline CapLayout cap_layout(int64_t n_rows, int64_t slots, int m, int n_groups) {
    CapLayout L;
    int64_t o = align256(slots * m * (int64_t)sizeof(Entry));
    L.len = o;
    o += align256(slots * 4);
    L.counts = o;
    o += align256(n_rows * n_groups);
    L.bound = o;
    o += align256(n_rows * (int64_t)sizeof(Entry));
    L.sat = o;
    o += align256(n_rows * (int64_t)sizeof(uint4));
    for (int i = 0; i < 2; ++i) {
        L.rows[i] = o;
        o += align256(n_rows * 4);
        L.users[i] = o;
        o += align256(n_rows * 4);
    }
    L.total = o;
    return L;
}

// The most (active row, slice) pairs any round over at most n_rows active rows can use: pick_slices depends on the rows only
// through their number of 64-row tiles.
inline int64_t max_slots(int64_t n_rows, int64_t n_cand_max, int per_sm, int slices) {
    int64_t best = 0;
    for (int64_t t = 1; t <= (n_rows + kRecUsers - 1) / kRecUsers; ++t) {
        const int64_t rows = t * kRecUsers < n_rows ? t * kRecUsers : n_rows;
        const int64_t v = rows * pick_slices(rows, n_cand_max, per_sm, slices);
        if (v > best) best = v;
    }
    return best;
}

// Dynamic shared memory of the score kernel at this width and k (opted in on the current device) and how many of its CTAs
// fit on one SM.  KGAT_ERR_UNSUPPORTED when one CTA does not fit.
template <bool kCapped>
int score_plan(const ConcatTables& T, int k, size_t* smem, int* per_sm) {
    *smem = score_smem_bytes(padded_width(T), k, kCapped);
    int dev = 0, max_smem = 0;
    KGAT_CUDA_TRY(cudaGetDevice(&dev));
    KGAT_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (*smem > (size_t)max_smem) return KGAT_ERR_UNSUPPORTED;
    KGAT_CUDA_TRY(cudaFuncSetAttribute(recommend_score_kernel<kCapped>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem));
    KGAT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, recommend_score_kernel<kCapped>, kRecThreads, *smem));
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
    if (score_plan<false>(T, k, &smem, &per_sm) != KGAT_OK) return -1;
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
    const int rc_plan = score_plan<false>(T, k, &smem, &per_sm);
    if (rc_plan != KGAT_OK) return rc_plan;
    const int S = pick_slices(n_users, n_cand_max, per_sm, slices);
    if (workspace_bytes_ < workspace_bytes(n_users, S, k)) return KGAT_ERR_WORKSPACE;
    ScoreParams<false> a;
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
    recommend_score_kernel<false><<<grid, kRecThreads, smem, s>>>(a);
    int rc = check_launch();
    if (rc != KGAT_OK) return rc;
    recommend_merge_kernel<<<(unsigned)((n_users * 32 + 255) / 256), 256, 0, s>>>(a.ws_list, a.ws_len, (int)n_users, S, k, cand_items, out_items,
                                                                                 out_scores, out_count);
    return check_launch();
}

int kgat_recommend_group_masks(const int32_t* row_ptr, const int32_t* col_idx, int64_t n_nodes, int32_t user_num, const int32_t* cand_items,
                               int64_t n_cand_max, const int32_t* n_cand, const int32_t* group_ptr, const int32_t* group_nodes, int32_t n_groups,
                               uint32_t* masks, void* stream) {
    if (n_nodes < 0 || n_nodes > 0x7fffffff || user_num < 0 || n_cand_max < 0 || n_cand_max > 0x7fffffff || n_groups < 0 || n_groups > kCapMaxGroups)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (n_cand_max == 0) return KGAT_OK;
    if (!row_ptr || !col_idx || !group_ptr || (n_groups > 0 && !group_nodes) || !cand_items || !masks) return KGAT_ERR_INVALID_ARGUMENT;
    recommend_mask_kernel<<<(unsigned)((n_cand_max * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        row_ptr, col_idx, user_num, cand_items, (int)n_cand_max, n_cand, group_ptr, group_nodes, n_groups, reinterpret_cast<uint4*>(masks));
    return check_launch();
}

int64_t kgat_recommend_capped_workspace_bytes(const kgat_tables_t* tables, int64_t n_users, int64_t n_cand_max, int32_t n_groups, int32_t k,
                                              int32_t m, int32_t slices) {
    ConcatTables T;
    if (!tables_from(tables, &T) || n_users < 0 || n_cand_max < 0 || n_groups < 0 || n_groups > kCapMaxGroups || k < 1 || m < k ||
        m > kRecMaxK || slices < 0 || slices > kRecMaxSlices)
        return -1;
    size_t smem = 0;
    int per_sm = 1;
    if (score_plan<true>(T, m, &smem, &per_sm) != KGAT_OK) return -1;
    return cap_layout(n_users, max_slots(n_users, n_cand_max, per_sm, slices), m, n_groups).total;
}

int kgat_recommend_capped_round(const kgat_tables_t* tables, const int32_t* users, int64_t n_users, const int32_t* cand_items, int64_t n_cand_max,
                                const int32_t* n_cand, const uint32_t* masks, const int32_t* caps, int32_t n_groups, int32_t k, int32_t m,
                                const int32_t* exclude_ptr, const int32_t* exclude_items, int32_t slices, int32_t round, int64_t n_active,
                                int32_t* n_active_next, int64_t* out_items, float* out_scores, int32_t* out_count, void* workspace,
                                int64_t workspace_bytes_, void* stream) {
    ConcatTables T;
    if (!tables_from(tables, &T) || n_users < 0 || n_users > 0x7fffffff || n_cand_max < 0 || n_cand_max > 0x7fffffff || n_groups < 0 ||
        n_groups > kCapMaxGroups || k < 1 || m < k || m > kRecMaxK || slices < 0 || slices > kRecMaxSlices || round < 0 || n_active < 0 ||
        n_active > n_users || (round == 0 && n_active != n_users))
        return KGAT_ERR_INVALID_ARGUMENT;
    if (n_active == 0) return KGAT_OK;
    if (!users || (n_cand_max > 0 && (!cand_items || !masks)) || (n_groups > 0 && !caps) || (exclude_ptr && !exclude_items) || !n_active_next ||
        !out_items || !out_scores || !out_count || !workspace)
        return KGAT_ERR_INVALID_ARGUMENT;
    size_t smem = 0;
    int per_sm = 1;
    const int rc_plan = score_plan<true>(T, m, &smem, &per_sm);
    if (rc_plan != KGAT_OK) return rc_plan;
    const CapLayout L = cap_layout(n_users, max_slots(n_users, n_cand_max, per_sm, slices), m, n_groups);
    if (workspace_bytes_ < L.total) return KGAT_ERR_WORKSPACE;
    const int S = pick_slices(n_active, n_cand_max, per_sm, slices);
    char* w = static_cast<char*>(workspace);
    const int in = (round + 1) & 1, out = round & 1;  // round r reads the list round r - 1 wrote
    ScoreParams<true> a;
    a.T = T;
    a.width_pad = padded_width(T);
    a.users = round == 0 ? users : reinterpret_cast<const int32_t*>(w + L.users[in]);
    a.n_users = (int)n_active;
    a.cand = cand_items;
    a.n_cand_max = (int)n_cand_max;
    a.n_cand_dev = n_cand;
    a.k = m;
    a.excl_ptr = exclude_ptr;
    a.excl_items = exclude_items;
    a.slices = S;
    a.ws_list = reinterpret_cast<Entry*>(w);
    a.ws_len = reinterpret_cast<int32_t*>(w + L.len);
    a.cap.rows = round == 0 ? nullptr : reinterpret_cast<const int32_t*>(w + L.rows[in]);
    a.cap.bound = reinterpret_cast<const Entry*>(w + L.bound);
    a.cap.sat = reinterpret_cast<const uint4*>(w + L.sat);
    a.cap.mask = reinterpret_cast<const uint4*>(masks);
    a.cap.caps = caps;
    a.cap.n_groups = n_groups;
    cudaStream_t s = (cudaStream_t)stream;
    KGAT_CUDA_TRY(cudaMemsetAsync(n_active_next, 0, sizeof(int32_t), s));
    const dim3 grid((unsigned)((n_active + kRecUsers - 1) / kRecUsers), (unsigned)S);
    recommend_score_kernel<true><<<grid, kRecThreads, smem, s>>>(a);
    int rc = check_launch();
    if (rc != KGAT_OK) return rc;
    GreedyArgs g;
    g.ws_list = a.ws_list;
    g.ws_len = a.ws_len;
    g.slices = S;
    g.m = m;
    g.k = k;
    g.n_active = (int)n_active;
    g.n_groups = n_groups;
    g.rows_in = a.cap.rows;
    g.users = users;
    g.cand = cand_items;
    g.mask = a.cap.mask;
    g.caps = caps;
    g.counts = reinterpret_cast<uint8_t*>(w + L.counts);
    g.bound = reinterpret_cast<Entry*>(w + L.bound);
    g.sat = reinterpret_cast<uint4*>(w + L.sat);
    g.rows_out = reinterpret_cast<int32_t*>(w + L.rows[out]);
    g.users_out = reinterpret_cast<int32_t*>(w + L.users[out]);
    g.n_out = n_active_next;
    g.out_items = out_items;
    g.out_scores = out_scores;
    g.out_count = out_count;
    recommend_capped_greedy_kernel<<<(unsigned)((n_active * 32 + 255) / 256), 256, 0, s>>>(g);
    return check_launch();
}

}  // extern "C"
