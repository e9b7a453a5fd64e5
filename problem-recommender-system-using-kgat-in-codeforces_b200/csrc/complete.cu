// Knowledge-graph completion with the trained TransR half (DESIGN section 4.9): the top-k tails of (h, r, ?) queries and the
// exact filtered rank of a known tail, without materialising an energy matrix.
//
// Energy E(h, r, t) = ||e_h W_r + e_r - e_t W_r||^2, bit-identical to the per-sample term of transr_fwd_kernel (losses.cu):
//   * x = e W_r: column c is (((0 + p0) + p1) + p2) + p3, p_w the sequential fmaf chain from +0 over rows [w D/4, (w+1) D/4)
//     of W_r (transr_partial / transr_combine);
//   * d = (x_h + e_r) - x_t;
//   * lane l's partial: the fmaf(d, d, .) chain from +0 over the columns K/32 l .. K/32 l + K/32 - 1;
//   * warp_sum's xor butterfly over the 32 lane partials: a balanced tree over the lanes in bit-reversed order, evaluated
//     here by one thread in a streaming pass that keeps one pending sum per tree level.
// Order: lower energy first.  Entries hold s = -E (a NaN energy stays a positive NaN, so it ranks first), so the key
// (float_key(s) << 32) | (0xFFFFFFFF - position) is recommend's order (common.cuh: beats) and the shared top-k helpers apply.
//
//   complete_project_kernel  out[g][i] = e_{ids[i]} W_r (+ e_r), one thread per output column;
//   complete_energy_kernel   E of (query, target) pairs from their projections;
//   complete_tile_kernel     one CTA per (64-query tile of one relation, candidate slice): the tile's query vectors and a
//       64-candidate tile of projections sit in shared memory, a thread owns 4 x 4 (query, candidate) pairs.  TOPK: every
//       query keeps a running top-k (a pair enters the pending buffer only when it beats the k-th entry and is not excluded);
//       COUNT: a pair counts when its key beats the target's and it is not excluded, one integer atomic per query and tile;
//   complete_merge_kernel    one warp per query merges the slices' lists (merge_slices);
//   complete_finalize_kernel one warp per query: rank (-1 for a target outside the candidates) and eligible candidates.
#include "common.cuh"

namespace kgat {
namespace {

constexpr int kCmpThreads = kTileThreads;
constexpr int kCmpQueries = kTileUsers;  // queries per CTA
constexpr int kCmpItems = kTileItems;    // candidates per tile
constexpr int kCmpMaxGroup = 32;         // relations projected at once
constexpr int64_t kCmpProjCap = 1LL << 30;  // bytes of candidate projections held at once

inline int64_t align256(int64_t b) { return (b + 255) & ~int64_t(255); }

// -E by its sign bit; any NaN becomes the positive NaN, whose float_key is the largest
__device__ __forceinline__ float neg_energy(float e) { return e != e ? __int_as_float(0x7fffffff) : __int_as_float(__float_as_int(e) ^ 0x80000000); }

__device__ __forceinline__ uint64_t complete_key(float e, int pos) {
    return ((uint64_t)float_key(neg_energy(e)) << 32) | (0xFFFFFFFFu - (uint32_t)pos);
}

// first position in p[0, n) whose value is >= x (p ascending)
__device__ __forceinline__ int64_t lower_bound_i64(const int64_t* __restrict__ p, int64_t n, int64_t x) {
    int64_t lo = 0;
    while (n > 0) {
        const int64_t half = n >> 1;
        if (__ldg(p + lo + half) < x) {
            lo += half + 1;
            n -= half + 1;
        } else {
            n = half;
        }
    }
    return lo;
}

// ---------------------------------------------------------------------------------------------------------------------
// projections
// ---------------------------------------------------------------------------------------------------------------------
// out[g][i][c] = (e_{ids[i]} W_r)[c] (+ e_r[c] when add_rel), r = rel_per_row ? rels[i] : rels[g]; grid (ceil(n K / 256), groups)
template <int DM, int KM>
__global__ void __launch_bounds__(256) complete_project_kernel(const float* __restrict__ emb, const float* __restrict__ rel_emb,
                                                               const float* __restrict__ W, const int32_t* __restrict__ ids, int n,
                                                               const int32_t* __restrict__ rels, bool rel_per_row, bool add_rel,
                                                               float* __restrict__ out) {
    constexpr int D = DM * 32, K = KM * 32, JW = D / 4;
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= (int64_t)n * K) return;
    const int i = (int)(e / K), c = (int)(e % K);
    const int64_t r = rel_per_row ? rels[i] : rels[blockIdx.y];
    const float* x = emb + (int64_t)ids[i] * D;
    const float* Wr = W + r * D * K + c;
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        float p = 0.f;
#pragma unroll 8
        for (int jj = 0; jj < JW; ++jj) p = fmaf(__ldg(x + w * JW + jj), __ldg(Wr + (int64_t)(w * JW + jj) * K), p);
        sum += p;
    }
    if (add_rel) sum = sum + __ldg(rel_emb + r * K + c);
    out[(int64_t)blockIdx.y * n * K + e] = sum;
}

// lane l's partial over d = q - x: the fmaf chain over columns KM l .. KM l + KM - 1
template <int KM>
__device__ __forceinline__ float lane_partial(const float* q, const float* x, int l) {
    float s = 0.f;
#pragma unroll
    for (int m = 0; m < KM; ++m) {
        const float d = q[KM * l + m] - x[KM * l + m];
        s = fmaf(d, d, s);
    }
    return s;
}

__host__ __device__ constexpr int brev5(int i) { return ((i & 1) << 4) | ((i & 2) << 2) | (i & 4) | ((i & 8) >> 2) | ((i & 16) >> 4); }

// E[i] = energy of query vector q[i] (= x_h + e_r) and tail projection x[i]; one thread per pair
template <int KM>
__global__ void __launch_bounds__(256) complete_energy_kernel(const float* __restrict__ q, const float* __restrict__ x, int n,
                                                              float* __restrict__ E) {
    constexpr int K = KM * 32;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* qi = q + (int64_t)i * K;
    const float* xi = x + (int64_t)i * K;
    float st[5];
#pragma unroll
    for (int t = 0; t < 32; ++t) {
        float v = lane_partial<KM>(qi, xi, brev5(t));
        int lvl = 0;
#pragma unroll
        for (; lvl < 5 && ((t >> lvl) & 1); ++lvl) v = st[lvl] + v;
        if (lvl < 5) st[lvl] = v;
        else E[i] = v;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// score tiles
// ---------------------------------------------------------------------------------------------------------------------
struct GroupTiles {
    int n;                      // relations of this launch
    int tile_ptr[kCmpMaxGroup + 1];  // CTA rows [tile_ptr[g], tile_ptr[g+1]) serve relation g
    int q_begin[kCmpMaxGroup];  // its queries [q_begin[g], q_end[g]) in sorted order
    int q_end[kCmpMaxGroup];
};

struct TileArgs {
    GroupTiles G;
    const float* qv;        // [n_q][K] query vectors, sorted by relation
    const int32_t* q_head;  // [n_q] head node of each sorted query
    const int32_t* q_rel;   // [n_q] its relation
    float* proj;            // [G.n][n_cand][K] candidate projections of this launch's relations
    const int32_t* cand;    // [n_cand] node ids; position = index
    int n_cand;
    const int64_t* ex_keys;  // nullable: known triples (h R + r) N + t, ascending
    int64_t n_ex;
    int64_t n_nodes, n_rel;
    int slices;
    int k;
    Entry* ws_list;          // TOPK: [n_q][slices][k]
    int32_t* ws_len;         // TOPK: [n_q][slices]
    const uint64_t* t_key;   // COUNT: [n_q] the target's key (all ones: nothing counts)
    unsigned long long* cnt;  // COUNT: [n_q]
};

inline size_t tile_smem_bytes(int K, int k, bool count) {
    size_t b = sizeof(float) * 2 * (size_t)K * kTilePad;
    if (!count) b += sizeof(Entry) * (size_t)kCmpQueries * (k + kCmpItems) + 2 * sizeof(int) * kCmpQueries;
    return b;
}

template <int KM, bool COUNT>
__global__ void __launch_bounds__(kCmpThreads, 1) complete_tile_kernel(TileArgs a) {
    constexpr int K = KM * 32;
    extern __shared__ float4 smem_f4[];
    float* Qs = reinterpret_cast<float*>(smem_f4);  // [K][kTilePad]: the tile's query vectors, transposed
    float* Cs = Qs + K * kTilePad;                  // [K][kTilePad]: one candidate tile's projections, transposed
    Entry* top = reinterpret_cast<Entry*>(Cs + K * kTilePad);  // TOPK: [kCmpQueries][k], sorted best-first
    Entry* pend = top + kCmpQueries * a.k;                     // TOPK: [kCmpQueries][kCmpItems], unordered
    int* n_top = reinterpret_cast<int*>(pend + kCmpQueries * kCmpItems);
    int* n_pend = n_top + kCmpQueries;

    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16, lane = tid & 31, warp = tid >> 5;
    int g = 0;
    while (g + 1 < a.G.n && (int)blockIdx.x >= a.G.tile_ptr[g + 1]) ++g;
    const int q0 = a.G.q_begin[g] + ((int)blockIdx.x - a.G.tile_ptr[g]) * kCmpQueries;
    const int nq = min(kCmpQueries, a.G.q_end[g] - q0);
    const int slice = blockIdx.y, k = a.k;
    const int c_begin = (int)((int64_t)a.n_cand * slice / a.slices), c_end = (int)((int64_t)a.n_cand * (slice + 1) / a.slices);
    const float* P = a.proj + (int64_t)g * a.n_cand * K;

    for (int e = tid; e < kCmpQueries * (K / 4); e += kCmpThreads) {
        const int r = e % kCmpQueries, q4 = e / kCmpQueries;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < nq) v = ldg4(a.qv + (int64_t)(q0 + r) * K + 4 * q4);
        Qs[(4 * q4 + 0) * kTilePad + r] = v.x;
        Qs[(4 * q4 + 1) * kTilePad + r] = v.y;
        Qs[(4 * q4 + 2) * kTilePad + r] = v.z;
        Qs[(4 * q4 + 3) * kTilePad + r] = v.w;
    }
    if (!COUNT && tid < kCmpQueries) { n_top[tid] = 0; n_pend[tid] = 0; }

    // per-thread known-triple ranges and target keys of its 4 queries
    int64_t ex_b[4], ex_n[4], base[4];
    uint64_t tk[4];
    int my_cnt[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int ql = ty * 4 + i;
        ex_b[i] = ex_n[i] = base[i] = 0;
        tk[i] = ~0ull;
        my_cnt[i] = 0;
        if (ql < nq) {
            base[i] = ((int64_t)a.q_head[q0 + ql] * a.n_rel + a.q_rel[q0 + ql]) * a.n_nodes;
            if (a.ex_keys) {
                ex_b[i] = lower_bound_i64(a.ex_keys, a.n_ex, base[i]);
                ex_n[i] = lower_bound_i64(a.ex_keys + ex_b[i], a.n_ex - ex_b[i], base[i] + a.n_nodes);
            }
            if (COUNT) tk[i] = a.t_key[q0 + ql];
        }
    }

    for (int c0 = c_begin; c0 < c_end; c0 += kCmpItems) {
        __syncthreads();  // the previous tile's projections (and, first, nothing) are no longer read
        for (int e = tid; e < kCmpItems * (K / 4); e += kCmpThreads) {
            const int r = e % kCmpItems, q4 = e / kCmpItems;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c0 + r < c_end) v = ldg4(P + (int64_t)(c0 + r) * K + 4 * q4);
            Cs[(4 * q4 + 0) * kTilePad + r] = v.x;
            Cs[(4 * q4 + 1) * kTilePad + r] = v.y;
            Cs[(4 * q4 + 2) * kTilePad + r] = v.z;
            Cs[(4 * q4 + 3) * kTilePad + r] = v.w;
        }
        __syncthreads();
        // energies of the 4 x 4 pairs: lane partials in bit-reversed lane order, folded into the butterfly's tree
        float E[4][4], st[5][4][4];
#pragma unroll
        for (int t = 0; t < 32; ++t) {
            const int l = brev5(t);
            float v[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) v[i][j] = 0.f;
#pragma unroll
            for (int m = 0; m < KM; ++m) {
                const float4 qv = *reinterpret_cast<const float4*>(&Qs[(KM * l + m) * kTilePad + ty * 4]);
                const float4 cv = *reinterpret_cast<const float4*>(&Cs[(KM * l + m) * kTilePad + tx * 4]);
                const float qr[4] = {qv.x, qv.y, qv.z, qv.w}, cr[4] = {cv.x, cv.y, cv.z, cv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float d = qr[i] - cr[j];
                        v[i][j] = fmaf(d, d, v[i][j]);
                    }
            }
            int lvl = 0;
#pragma unroll
            for (; lvl < 5 && ((t >> lvl) & 1); ++lvl)
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[i][j] = st[lvl][i][j] + v[i][j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (lvl < 5) st[lvl][i][j] = v[i][j];
                    else E[i][j] = v[i][j];
                }
        }

        if (COUNT) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (ty * 4 + i >= nq) continue;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int c = c0 + tx * 4 + j;
                    if (c >= c_end || complete_key(E[i][j], c) <= tk[i]) continue;
                    if (ex_n[i] > 0) {
                        const int64_t key = base[i] + a.cand[c];
                        const int64_t p = lower_bound_i64(a.ex_keys + ex_b[i], ex_n[i], key);
                        if (p < ex_n[i] && a.ex_keys[ex_b[i] + p] == key) continue;
                    }
                    ++my_cnt[i];
                }
            }
            continue;
        }

        // admission: beats the query's k-th entry (or the list is not full) and is not a known triple
        bool any = false;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int ql = ty * 4 + i;
            if (ql >= nq) continue;
            const int nt = n_top[ql];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const Entry x{neg_energy(E[i][j]), c0 + tx * 4 + j};
                if (x.c >= c_end) continue;
                if (nt == k && !beats(x, top[ql * k + k - 1])) continue;
                if (ex_n[i] > 0) {
                    const int64_t key = base[i] + a.cand[x.c];
                    const int64_t p = lower_bound_i64(a.ex_keys + ex_b[i], ex_n[i], key);
                    if (p < ex_n[i] && a.ex_keys[ex_b[i] + p] == key) continue;
                }
                pend[ql * kCmpItems + atomicAdd(&n_pend[ql], 1)] = x;
                any = true;
            }
        }
        if (!__syncthreads_or(any)) continue;
        for (int ql = warp; ql < kCmpQueries; ql += kCmpThreads / 32) {
            const int np = n_pend[ql];
            if (np == 0) continue;
            const int n_new = fold_pending(top + ql * k, n_top[ql], pend + ql * kCmpItems, np, k, lane);
            if (lane == 0) {
                n_top[ql] = n_new;
                n_pend[ql] = 0;
            }
            __syncwarp();
        }
    }

    if (COUNT) {
        // the 16 threads of a query row sit in one half-warp: sum there, one atomic per query and tile
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int v = my_cnt[i];
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
            if (tx == 0 && ty * 4 + i < nq && v > 0) atomicAdd(a.cnt + q0 + ty * 4 + i, (unsigned long long)v);
        }
        return;
    }
    __syncthreads();
    for (int ql = warp; ql < nq; ql += kCmpThreads / 32) {
        const int nt = n_top[ql];
        const int64_t o = (int64_t)(q0 + ql) * a.slices + slice;
        for (int i = lane; i < nt; i += 32) a.ws_list[o * k + i] = top[ql * k + i];
        if (lane == 0) a.ws_len[o] = nt;
    }
}

// One warp per sorted query; row q_out[q] of the outputs.
__global__ void __launch_bounds__(256) complete_merge_kernel(const Entry* __restrict__ ws_list, const int32_t* __restrict__ ws_len, int n_q,
                                                             int slices, int k, const int32_t* __restrict__ q_out,
                                                             const int32_t* __restrict__ cand, int64_t* __restrict__ out_tails,
                                                             float* __restrict__ out_energy, int32_t* __restrict__ out_count) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (q >= n_q) return;
    const int64_t row = q_out[q];
    const int total = merge_slices(ws_list + q * slices * k, ws_len + q * slices, slices, k, lane, [&](int r, const Entry& x) {
        out_tails[row * k + r] = cand[x.c];
        out_energy[row * k + r] = neg_energy(x.s);
    });
    for (int r = total + lane; r < k; r += 32) {
        out_tails[row * k + r] = -1;
        out_energy[row * k + r] = INFINITY;
    }
    if (lane == 0) out_count[row] = total;
}

// One thread per sorted query: the target's key from its energy and position (all ones when it is not a candidate).
__global__ void __launch_bounds__(256) complete_target_key_kernel(const float* __restrict__ E, const int32_t* __restrict__ tails, int n_q,
                                                                  const int32_t* __restrict__ pos_map, int n_cand, uint64_t* __restrict__ t_key,
                                                                  unsigned long long* __restrict__ cnt) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_q) return;
    const int t = tails[q];
    const int pos = pos_map ? pos_map[t] : (t < n_cand ? t : -1);
    t_key[q] = pos >= 0 ? complete_key(E[q], pos) : ~0ull;
    cnt[q] = 0;
}

// One warp per sorted query: rank and eligible candidates (known triples (h, r, c) of a candidate c != t are not eligible).
__global__ void __launch_bounds__(256) complete_finalize_kernel(const int32_t* __restrict__ heads, const int32_t* __restrict__ rels,
                                                                const int32_t* __restrict__ tails, int n_q, const int32_t* __restrict__ q_out,
                                                                const int32_t* __restrict__ pos_map, int n_cand, const int64_t* __restrict__ ex_keys,
                                                                int64_t n_ex, int64_t n_nodes, int64_t n_rel, const uint64_t* __restrict__ t_key,
                                                                const unsigned long long* __restrict__ cnt, const float* __restrict__ E,
                                                                float* __restrict__ out_energy, int64_t* __restrict__ out_rank,
                                                                int64_t* __restrict__ out_eligible) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (q >= n_q) return;
    const int t = tails[q];
    int excluded = 0;
    if (ex_keys) {
        const int64_t base = ((int64_t)heads[q] * n_rel + rels[q]) * n_nodes;
        const int64_t b = lower_bound_i64(ex_keys, n_ex, base);
        const int64_t e = b + lower_bound_i64(ex_keys + b, n_ex - b, base + n_nodes);
        for (int64_t i = b + lane; i < e; i += 32) {
            const int c = (int)(ex_keys[i] - base);
            const int pos = pos_map ? pos_map[c] : (c < n_cand ? c : -1);
            excluded += c != t && pos >= 0;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) excluded += __shfl_xor_sync(kFull, excluded, o);
    if (lane == 0) {
        const int64_t row = q_out[q];
        out_energy[row] = E[q];
        out_rank[row] = t_key[q] == ~0ull ? -1 : (int64_t)cnt[q];
        out_eligible[row] = (int64_t)n_cand - excluded;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
struct Plan {
    int K;
    size_t smem;
    int per_sm;
    int slices;
    int group;        // relations per candidate projection pass
    int64_t q_bytes, t_bytes, proj_bytes, list_bytes, len_bytes, key_bytes, cnt_bytes;
    int64_t total() const { return q_bytes + t_bytes + proj_bytes + list_bytes + len_bytes + key_bytes + cnt_bytes; }
};

template <int KM, bool COUNT>
int tile_occupancy(size_t smem, int* per_sm) {
    KGAT_CUDA_TRY(cudaFuncSetAttribute(complete_tile_kernel<KM, COUNT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    KGAT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, complete_tile_kernel<KM, COUNT>, kCmpThreads, smem));
    return KGAT_OK;
}

// n_tiles: 64-query tiles over all relations; count: kg_rank (k unused) or complete
int make_plan(int d, int kdim, int64_t n_q, int64_t n_tiles, int64_t n_cand, int32_t n_rel_used, int k, int slices, bool count, Plan* p) {
    if (!((d == 32 && kdim == 32) || (d == 64 && kdim == 64) || (d == 128 && kdim == 128))) return KGAT_ERR_UNSUPPORTED;
    if (n_q < 0 || n_q > 0x7fffffff || n_tiles < 0 || n_cand < 0 || n_cand > 0x7fffffff || n_rel_used < 0 || slices < 0 ||
        slices > kTileMaxSlices || (!count && (k < 1 || k > kTopkMaxK)))
        return KGAT_ERR_INVALID_ARGUMENT;
    p->K = kdim;
    p->smem = tile_smem_bytes(kdim, k, count);
    int dev = 0, max_smem = 0;
    KGAT_CUDA_TRY(cudaGetDevice(&dev));
    KGAT_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (p->smem > (size_t)max_smem) return KGAT_ERR_UNSUPPORTED;
    p->per_sm = 1;
    int rc = KGAT_OK;
    if (kdim == 32) rc = count ? tile_occupancy<1, true>(p->smem, &p->per_sm) : tile_occupancy<1, false>(p->smem, &p->per_sm);
    else if (kdim == 64) rc = count ? tile_occupancy<2, true>(p->smem, &p->per_sm) : tile_occupancy<2, false>(p->smem, &p->per_sm);
    else rc = count ? tile_occupancy<4, true>(p->smem, &p->per_sm) : tile_occupancy<4, false>(p->smem, &p->per_sm);
    if (rc != KGAT_OK) return rc;
    if (p->per_sm < 1) p->per_sm = 1;
    p->slices = pick_slices(n_tiles * kCmpQueries, n_cand, p->per_sm, slices);
    const int64_t per_rel = n_cand * kdim * (int64_t)sizeof(float);
    int64_t grp = per_rel > 0 ? kCmpProjCap / per_rel : kCmpMaxGroup;
    if (grp > kCmpMaxGroup) grp = kCmpMaxGroup;
    if (grp > n_rel_used) grp = n_rel_used;
    p->group = (int)(grp < 1 ? 1 : grp);
    p->q_bytes = align256(n_q * kdim * 4);
    p->t_bytes = count ? align256(n_q * kdim * 4) + align256(n_q * 4) : 0;  // target projections, energies
    p->proj_bytes = align256(p->group * per_rel);
    p->list_bytes = count ? 0 : align256(n_q * p->slices * (int64_t)k * sizeof(Entry));
    p->len_bytes = count ? 0 : align256(n_q * p->slices * 4);
    p->key_bytes = count ? align256(n_q * 8) : 0;
    p->cnt_bytes = count ? align256(n_q * 8) : 0;
    return KGAT_OK;
}

#define KGAT_COMPLETE_DISPATCH(CALL)                                          \
    if (kdim == 32) { constexpr int DM = 1, KM = 1; (void)DM; CALL; }         \
    else if (kdim == 64) { constexpr int DM = 2, KM = 2; (void)DM; CALL; }   \
    else { constexpr int DM = 4, KM = 4; (void)DM; CALL; }

int project(const float* emb, const float* rel_emb, const float* W, int kdim, const int32_t* ids, int n, const int32_t* rels, int groups,
            bool rel_per_row, bool add_rel, float* out, cudaStream_t s) {
    if (n == 0) return KGAT_OK;
    const dim3 grid((unsigned)(((int64_t)n * kdim + 255) / 256), (unsigned)groups);
    KGAT_COMPLETE_DISPATCH((complete_project_kernel<DM, KM><<<grid, 256, 0, s>>>(emb, rel_emb, W, ids, n, rels, rel_per_row, add_rel, out)));
    return check_launch();
}

// The tile launches, relation group by relation group: project the candidates under the group's relations, then score.
template <bool COUNT>
int run_tiles(const Plan& p, TileArgs a, const float* emb, const float* rel_emb, const float* W, const int64_t* seg_ptr_host, int n_seg,
              const int32_t* seg_rel, cudaStream_t s) {
    const int kdim = p.K;
    for (int g0 = 0; g0 < n_seg; g0 += p.group) {
        const int ng = n_seg - g0 < p.group ? n_seg - g0 : p.group;
        GroupTiles G;
        G.n = ng;
        G.tile_ptr[0] = 0;
        for (int g = 0; g < ng; ++g) {
            G.q_begin[g] = (int)seg_ptr_host[g0 + g];
            G.q_end[g] = (int)seg_ptr_host[g0 + g + 1];
            G.tile_ptr[g + 1] = G.tile_ptr[g] + (G.q_end[g] - G.q_begin[g] + kCmpQueries - 1) / kCmpQueries;
        }
        if (G.tile_ptr[ng] == 0 || a.n_cand == 0) continue;
        int rc = project(emb, rel_emb, W, kdim, a.cand, a.n_cand, seg_rel + g0, ng, false, false, a.proj, s);
        if (rc != KGAT_OK) return rc;
        a.G = G;
        const dim3 grid((unsigned)G.tile_ptr[ng], (unsigned)a.slices);
        KGAT_COMPLETE_DISPATCH((complete_tile_kernel<KM, COUNT><<<grid, kCmpThreads, p.smem, s>>>(a)));
        rc = check_launch();
        if (rc != KGAT_OK) return rc;
    }
    return KGAT_OK;
}

// checks shared by both entry points; n_tiles from the host segment table
int check_segments(const int64_t* seg_ptr_host, int n_seg, int64_t n_q, int64_t* n_tiles) {
    if (n_seg < 0 || (n_seg > 0 && !seg_ptr_host)) return KGAT_ERR_INVALID_ARGUMENT;
    *n_tiles = 0;
    if (n_seg == 0) return n_q == 0 ? KGAT_OK : KGAT_ERR_INVALID_ARGUMENT;
    if (seg_ptr_host[0] != 0 || seg_ptr_host[n_seg] != n_q) return KGAT_ERR_INVALID_ARGUMENT;
    for (int g = 0; g < n_seg; ++g) {
        if (seg_ptr_host[g + 1] <= seg_ptr_host[g]) return KGAT_ERR_INVALID_ARGUMENT;
        *n_tiles += (seg_ptr_host[g + 1] - seg_ptr_host[g] + kCmpQueries - 1) / kCmpQueries;
    }
    return KGAT_OK;
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int64_t kgat_complete_workspace_bytes(int32_t d, int32_t kdim, int64_t n_queries, int64_t n_tiles, int64_t n_cand, int32_t n_rel_used, int32_t k,
                                      int32_t slices, int32_t count) {
    Plan p;
    if (make_plan(d, kdim, n_queries, n_tiles, n_cand, n_rel_used, k, slices, count != 0, &p) != KGAT_OK) return -1;
    return p.total();
}

int kgat_complete_topk(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t kdim, int64_t n_nodes, int64_t n_rel,
                       const int32_t* heads, const int32_t* rels, const int32_t* q_out, int64_t n_q, const int64_t* seg_ptr_host,
                       const int32_t* seg_rel, int32_t n_seg, const int32_t* cand, int64_t n_cand,
                       const int64_t* ex_keys, int64_t n_ex, int32_t k, int32_t slices, int64_t* out_tails, float* out_energy,
                       int32_t* out_count, void* workspace, int64_t workspace_bytes, void* stream) {
    int64_t n_tiles = 0;
    int rc = check_segments(seg_ptr_host, n_seg, n_q, &n_tiles);
    if (rc != KGAT_OK) return rc;
    Plan p;
    rc = make_plan(d, kdim, n_q, n_tiles, n_cand, n_seg, k, slices, false, &p);
    if (rc != KGAT_OK) return rc;
    if (n_q == 0) return KGAT_OK;
    if (!emb || !rel_emb || !W || !heads || !rels || !q_out || !seg_rel || (n_cand > 0 && !cand) || (n_ex > 0 && !ex_keys) || n_ex < 0 ||
        n_nodes <= 0 || n_rel <= 0 || !out_tails || !out_energy || !out_count || !workspace)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < p.total()) return KGAT_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    char* w = static_cast<char*>(workspace);
    float* qv = reinterpret_cast<float*>(w);
    TileArgs a{};
    a.qv = qv;
    a.q_head = heads;
    a.q_rel = rels;
    a.proj = reinterpret_cast<float*>(w + p.q_bytes + p.t_bytes);
    a.cand = cand;
    a.n_cand = (int)n_cand;
    a.ex_keys = n_ex > 0 ? ex_keys : nullptr;
    a.n_ex = n_ex;
    a.n_nodes = n_nodes;
    a.n_rel = n_rel;
    a.slices = p.slices;
    a.k = k;
    a.ws_list = reinterpret_cast<Entry*>(w + p.q_bytes + p.t_bytes + p.proj_bytes);
    a.ws_len = reinterpret_cast<int32_t*>(w + p.q_bytes + p.t_bytes + p.proj_bytes + p.list_bytes);
    rc = project(emb, rel_emb, W, kdim, heads, (int)n_q, rels, 1, true, true, qv, s);
    if (rc != KGAT_OK) return rc;
    if (n_cand == 0) {
        KGAT_CUDA_TRY(cudaMemsetAsync(a.ws_len, 0, n_q * p.slices * 4, s));
    } else {
        rc = run_tiles<false>(p, a, emb, rel_emb, W, seg_ptr_host, n_seg, seg_rel, s);
        if (rc != KGAT_OK) return rc;
    }
    complete_merge_kernel<<<(unsigned)((n_q * 32 + 255) / 256), 256, 0, s>>>(a.ws_list, a.ws_len, (int)n_q, p.slices, k, q_out, cand, out_tails,
                                                                            out_energy, out_count);
    return check_launch();
}

int kgat_complete_rank(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t kdim, int64_t n_nodes, int64_t n_rel,
                       const int32_t* heads, const int32_t* rels, const int32_t* tails, const int32_t* q_out, int64_t n_q,
                       const int64_t* seg_ptr_host, const int32_t* seg_rel, int32_t n_seg,
                       const int32_t* cand, int64_t n_cand, const int32_t* pos_map, const int64_t* ex_keys, int64_t n_ex, int32_t slices,
                       float* out_energy, int64_t* out_rank, int64_t* out_eligible, void* workspace, int64_t workspace_bytes, void* stream) {
    int64_t n_tiles = 0;
    int rc = check_segments(seg_ptr_host, n_seg, n_q, &n_tiles);
    if (rc != KGAT_OK) return rc;
    Plan p;
    rc = make_plan(d, kdim, n_q, n_tiles, n_cand, n_seg, 1, slices, true, &p);
    if (rc != KGAT_OK) return rc;
    if (n_q == 0) return KGAT_OK;
    if (!emb || !rel_emb || !W || !heads || !rels || !tails || !q_out || !seg_rel || (n_cand > 0 && !cand) || (n_ex > 0 && !ex_keys) ||
        n_ex < 0 || n_nodes <= 0 || n_rel <= 0 || !out_energy || !out_rank || !out_eligible || !workspace)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < p.total()) return KGAT_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    char* w = static_cast<char*>(workspace);
    float* qv = reinterpret_cast<float*>(w);
    float* xt = reinterpret_cast<float*>(w + p.q_bytes);
    float* E = reinterpret_cast<float*>(w + p.q_bytes + align256(n_q * kdim * 4));
    TileArgs a{};
    a.qv = qv;
    a.q_head = heads;
    a.q_rel = rels;
    a.proj = reinterpret_cast<float*>(w + p.q_bytes + p.t_bytes);
    a.cand = cand;
    a.n_cand = (int)n_cand;
    a.ex_keys = n_ex > 0 ? ex_keys : nullptr;
    a.n_ex = n_ex;
    a.n_nodes = n_nodes;
    a.n_rel = n_rel;
    a.slices = p.slices;
    a.t_key = reinterpret_cast<uint64_t*>(w + p.q_bytes + p.t_bytes + p.proj_bytes);
    a.cnt = reinterpret_cast<unsigned long long*>(w + p.q_bytes + p.t_bytes + p.proj_bytes + p.key_bytes);
    rc = project(emb, rel_emb, W, kdim, heads, (int)n_q, rels, 1, true, true, qv, s);
    if (rc != KGAT_OK) return rc;
    rc = project(emb, rel_emb, W, kdim, tails, (int)n_q, rels, 1, true, false, xt, s);
    if (rc != KGAT_OK) return rc;
    KGAT_COMPLETE_DISPATCH((complete_energy_kernel<KM><<<(unsigned)((n_q + 255) / 256), 256, 0, s>>>(qv, xt, (int)n_q, E)));
    rc = check_launch();
    if (rc != KGAT_OK) return rc;
    complete_target_key_kernel<<<(unsigned)((n_q + 255) / 256), 256, 0, s>>>(E, tails, (int)n_q, pos_map, (int)n_cand,
                                                                             const_cast<uint64_t*>(a.t_key), a.cnt);
    rc = check_launch();
    if (rc != KGAT_OK) return rc;
    rc = run_tiles<true>(p, a, emb, rel_emb, W, seg_ptr_host, n_seg, seg_rel, s);
    if (rc != KGAT_OK) return rc;
    complete_finalize_kernel<<<(unsigned)((n_q * 32 + 255) / 256), 256, 0, s>>>(heads, rels, tails, (int)n_q, q_out, pos_map, (int)n_cand, a.ex_keys,
                                                                               n_ex, n_nodes, n_rel, a.t_key, a.cnt, E, out_energy, out_rank,
                                                                               out_eligible);
    return check_launch();
}

}  // extern "C"
