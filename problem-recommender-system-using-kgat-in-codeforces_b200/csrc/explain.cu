// Path explanations: the top-k attention-weighted simple paths s -> ... -> t of up to 3 hops through the
// attentive matrix A, plus the number of such paths and their summed weight per length (DESIGN section 4.6).
//
// A path's weight is the left-to-right fp32 product of its hop values; paths rank by weight descending, then hop
// count ascending, then (v1, v2) ascending -- a total order, so the top-k set does not depend on the order in
// which candidates are found.
//
// Work of a pair: the 1-hop path is one binary search of t in row s; the 2-hop paths are row s INTERSECT In(t)
// (In(t) = row t of A^T); the 3-hop paths are, for every a in row s, row a INTERSECT In(t).  Every intersection
// takes each element of the shorter list and binary-searches it in the longer one, so a pair's work is
// T = min(deg s, |In t|) + sum_a min(deg a, |In t|) probes.  That flat probe range is cut into `units` equal
// slices, one CTA each (a hub pair is spread over many SMs); kernel 1 leaves each slice's own top-k list
// (sorted) and its per-length counts / fp64 weight sums in the workspace, kernel 2 merges a pair's lists and
// sums the partials in slice order, so `mass` is bitwise reproducible without float atomics.
#include "common.cuh"

namespace kgat {
namespace {

constexpr int kExplainThreads = 256;
constexpr int kExplainMaxK = 64;
constexpr int kExplainMaxHops = 3;

struct Cand {
    float w;
    int h;
    int v1, v2;
    int slot[3];
    int pad;
};
static_assert(sizeof(Cand) == 32, "Cand layout");

// true when path a ranks before path b
__device__ __forceinline__ bool beats(const Cand& a, const Cand& b) {
    if (a.w != b.w) return a.w > b.w;
    if (a.h != b.h) return a.h < b.h;
    if (a.v1 != b.v1) return a.v1 < b.v1;
    return a.v2 < b.v2;
}

int explain_units(int64_t n_pairs) {
    const int64_t u = 65536 / (n_pairs > 0 ? n_pairs : 1);
    return (int)(u < 8 ? 8 : (u > 64 ? 64 : u));
}

struct Workspace {
    Cand* cand;       // [n_units][k], each list sorted best-first
    int32_t* n_cand;  // [n_units]
    double* mass;     // [n_units][kExplainMaxHops]
    long long* count; // [n_units][kExplainMaxHops]
};

inline int64_t align256(int64_t b) { return (b + 255) & ~int64_t(255); }

Workspace carve(void* base, int64_t n_units, int k) {
    char* p = static_cast<char*>(base);
    Workspace w;
    w.cand = reinterpret_cast<Cand*>(p);
    p += align256(n_units * k * (int64_t)sizeof(Cand));
    w.n_cand = reinterpret_cast<int32_t*>(p);
    p += align256(n_units * 4);
    w.mass = reinterpret_cast<double*>(p);
    p += align256(n_units * kExplainMaxHops * 8);
    w.count = reinterpret_cast<long long*>(p);
    return w;
}

int64_t workspace_bytes(int64_t n_units, int k) {
    return align256(n_units * k * (int64_t)sizeof(Cand)) + align256(n_units * 4) + 2 * align256(n_units * kExplainMaxHops * 8);
}

struct Graph {
    const int32_t* __restrict__ row_ptr;
    const int32_t* __restrict__ col_idx;
    const float* __restrict__ vals;
    const int32_t* __restrict__ t_ptr;
    const int32_t* __restrict__ t_idx;
    const int32_t* __restrict__ t_perm;
    int64_t n;
};

struct ExplainSmem {
    Cand top[2][kExplainMaxK];
    Cand buf[kExplainThreads];
    long long pre[kExplainThreads];  // exclusive prefix of the tile's probe counts
    int item_row[kExplainThreads];   // row intersected with In(t): s for the 2-hop item, a for a 3-hop item
    int item_slot0[kExplainThreads]; // CSR slot of (s, a) for a 3-hop item
    long long warp_tot[kExplainThreads / 32];
    int warp_cnt[kExplainThreads / 32];
    int cur, ntop;
};

// exclusive block scan of v (all threads call); returns the block total through *total
__device__ long long block_exclusive_scan(long long v, ExplainSmem& sm, long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) sm.warp_tot[warp] = incl;
    __syncthreads();
    long long before = 0, tot = 0;
    for (int w = 0; w < kExplainThreads / 32; ++w) {
        if (w < warp) before += sm.warp_tot[w];
        tot += sm.warp_tot[w];
    }
    __syncthreads();
    *total = tot;
    return before + incl - v;
}

// Offers every thread's candidate (when `has`) to the CTA's running top-k.  Called by all threads.
__device__ void offer(bool has, const Cand& c, int k, ExplainSmem& sm) {
    const int ntop = sm.ntop, cur = sm.cur;
    const bool admit = has && (ntop < k || beats(c, sm.top[cur][ntop - 1]));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned bal = __ballot_sync(kFull, admit);
    if (lane == 0) sm.warp_cnt[warp] = __popc(bal);
    const int n_adm = __syncthreads_count(admit);
    if (n_adm == 0) return;
    if (admit) {
        int pos = __popc(bal & ((1u << lane) - 1));
        for (int w = 0; w < warp; ++w) pos += sm.warp_cnt[w];
        sm.buf[pos] = c;
    }
    __syncthreads();
    // rank selection over the union (a total order: every rank is distinct)
    const int n_union = ntop + n_adm;
    Cand* next = sm.top[cur ^ 1];
    for (int i = threadIdx.x; i < n_union; i += kExplainThreads) {
        const Cand x = i < ntop ? sm.top[cur][i] : sm.buf[i - ntop];
        int rank = 0;
        if (i < ntop) {
            rank = i;
        } else {
            int lo = 0, n = ntop;  // top is sorted: count its members that beat x
            while (n > 0) {
                const int half = n >> 1;
                if (beats(sm.top[cur][lo + half], x)) {
                    lo += half + 1;
                    n -= half + 1;
                } else {
                    n = half;
                }
            }
            rank = lo;
        }
        for (int j = 0; j < n_adm && rank < k; ++j) rank += beats(sm.buf[j], x);
        if (rank < k) next[rank] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        sm.cur = cur ^ 1;
        sm.ntop = n_union < k ? n_union : k;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kExplainThreads) explain_units_kernel(Graph g, const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                                                                        int units, int k, int H, Workspace ws) {
    __shared__ ExplainSmem sm;
    const int64_t unit = blockIdx.x;
    const int64_t pair = unit / units;
    const int u = (int)(unit % units);
    const int tid = threadIdx.x;
    if (tid == 0) { sm.cur = 0; sm.ntop = 0; }
    const int s = src[pair], t = dst[pair];
    const bool valid = s >= 0 && s < g.n && t >= 0 && t < g.n && s != t;
    long long cnt[kExplainMaxHops] = {0, 0, 0};
    double mass[kExplainMaxHops] = {0.0, 0.0, 0.0};
    __syncthreads();
    if (valid) {
        const int rb_s = g.row_ptr[s], deg_s = g.row_ptr[s + 1] - rb_s;
        const int tb = g.t_ptr[t], tl = g.t_ptr[t + 1] - tb;
        // 1 hop
        {
            Cand c;
            bool has = false;
            if (u == 0 && tid == 0) {
                const int p = lower_bound_i32(g.col_idx + rb_s, deg_s, t);
                if (p < deg_s && g.col_idx[rb_s + p] == t) {
                    c.w = g.vals[rb_s + p];
                    c.h = 1; c.v1 = t; c.v2 = -1;
                    c.slot[0] = rb_s + p; c.slot[1] = c.slot[2] = -1;
                    c.pad = 0;
                    has = true;
                    cnt[0] = 1;
                    mass[0] = (double)c.w;
                }
            }
            offer(has, c, k, sm);
        }
        // items: 0 = the 2-hop intersection row s & In(t); 1 + i = the 3-hop intersection row a_i & In(t), a_i = col_idx[rb_s + i]
        const int n_items = H >= 2 ? 1 + (H >= 3 ? deg_s : 0) : 0;
        auto item_len = [&](int item, int& row, int& slot0) -> long long {
            if (item == 0) {
                row = s; slot0 = -1;
                return deg_s < tl ? deg_s : tl;
            }
            slot0 = rb_s + item - 1;
            row = g.col_idx[slot0];
            if (row == s || row == t) return 0;
            const int d = g.row_ptr[row + 1] - g.row_ptr[row];
            return d < tl ? d : tl;
        };
        // pass 1: the pair's total probe count -> this unit's slice [lo, hi)
        long long mine = 0;
        for (int item = tid; item < n_items; item += kExplainThreads) {
            int row, slot0;
            mine += item_len(item, row, slot0);
        }
        long long total;
        block_exclusive_scan(mine, sm, &total);
        const long long lo = total * u / units, hi = total * (u + 1) / units;
        // pass 2: walk the items in tiles of one item per thread
        long long base = 0;
        for (int tile = 0; tile < n_items && base < hi; tile += kExplainThreads) {
            const int item = tile + tid;
            int row = -1, slot0 = -1;
            const long long len = item < n_items ? item_len(item, row, slot0) : 0;
            long long tile_tot;
            const long long ex = block_exclusive_scan(len, sm, &tile_tot);
            sm.pre[tid] = ex;
            sm.item_row[tid] = row;
            sm.item_slot0[tid] = slot0;
            __syncthreads();
            const long long f_begin = lo > base ? lo : base, f_end = hi < base + tile_tot ? hi : base + tile_tot;
            for (long long f0 = f_begin; f0 < f_end; f0 += kExplainThreads) {  // uniform trip count over the CTA
                const long long f = f0 + tid;
                Cand c;
                bool has = false;
                if (f < f_end) {
                    const long long off = f - base;
                    // the owner of `off` is the last item whose prefix is <= off (empty items before it share its prefix)
                    int lo_i = 0, n_i = kExplainThreads;
                    while (n_i > 1) {
                        const int half = n_i >> 1;
                        if (sm.pre[lo_i + half] <= off) { lo_i += half; n_i -= half; } else { n_i = half; }
                    }
                    const int j = (int)(off - sm.pre[lo_i]);
                    const int r = sm.item_row[lo_i];
                    const int rb = g.row_ptr[r], rl = g.row_ptr[r + 1] - rb;
                    int x, p1, p2;
                    bool match;
                    if (rl <= tl) {
                        p1 = j;
                        x = g.col_idx[rb + j];
                        p2 = lower_bound_i32(g.t_idx + tb, tl, x);
                        match = p2 < tl && g.t_idx[tb + p2] == x;
                    } else {
                        p2 = j;
                        x = g.t_idx[tb + j];
                        p1 = lower_bound_i32(g.col_idx + rb, rl, x);
                        match = p1 < rl && g.col_idx[rb + p1] == x;
                    }
                    if (match) {
                        const int item_idx = tile + lo_i;
                        c.pad = 0;
                        if (item_idx == 0) {  // s -> x -> t
                            if (x != s && x != t) {
                                c.h = 2; c.v1 = x; c.v2 = t;
                                c.slot[0] = rb + p1; c.slot[1] = g.t_perm[tb + p2]; c.slot[2] = -1;
                                c.w = __fmul_rn(g.vals[c.slot[0]], g.vals[c.slot[1]]);
                                has = true;
                            }
                        } else if (x != s && x != r && x != t) {  // s -> r -> x -> t
                            c.h = 3; c.v1 = r; c.v2 = x;
                            c.slot[0] = sm.item_slot0[lo_i]; c.slot[1] = rb + p1; c.slot[2] = g.t_perm[tb + p2];
                            c.w = __fmul_rn(__fmul_rn(g.vals[c.slot[0]], g.vals[c.slot[1]]), g.vals[c.slot[2]]);
                            has = true;
                        }
                        if (has) {
                            cnt[c.h - 1] += 1;
                            mass[c.h - 1] += (double)c.w;
                        }
                    }
                }
                offer(has, c, k, sm);
            }
            base += tile_tot;
            __syncthreads();  // pre / item arrays are rewritten by the next tile
        }
    }
    // this unit's list and partials (fixed-order block reduction: thread order within a warp, then warp order)
    const int n_top = sm.ntop, cur = sm.cur;
    for (int i = tid; i < n_top; i += kExplainThreads) ws.cand[unit * k + i] = sm.top[cur][i];
    if (tid == 0) ws.n_cand[unit] = n_top;
    for (int h = 0; h < kExplainMaxHops; ++h) {
        double m = mass[h];
        long long c = cnt[h];
        for (int o = 16; o > 0; o >>= 1) {
            m += __shfl_down_sync(kFull, m, o);
            c += __shfl_down_sync(kFull, c, o);
        }
        __shared__ double s_m[kExplainThreads / 32];
        __shared__ long long s_c[kExplainThreads / 32];
        if ((tid & 31) == 0) { s_m[tid >> 5] = m; s_c[tid >> 5] = c; }
        __syncthreads();
        if (tid == 0) {
            double tm = 0.0;
            long long tc = 0;
            for (int w = 0; w < kExplainThreads / 32; ++w) { tm += s_m[w]; tc += s_c[w]; }
            ws.mass[unit * kExplainMaxHops + h] = tm;
            ws.count[unit * kExplainMaxHops + h] = tc;
        }
        __syncthreads();
    }
}

// One CTA per pair: merge the units' sorted lists (rank = own index + members of the other lists that beat it), write the
// outputs with their padding, and sum the units' partials in unit order.
__global__ void __launch_bounds__(kExplainThreads) explain_merge_kernel(const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                                                                        int units, int k, int H, Workspace ws, int64_t* __restrict__ nodes,
                                                                        int64_t* __restrict__ slots, int32_t* __restrict__ hops,
                                                                        float* __restrict__ weight, int64_t* __restrict__ count,
                                                                        float* __restrict__ mass) {
    const int64_t pair = blockIdx.x;
    const int64_t u0 = pair * units;
    __shared__ int s_n[64];
    __shared__ int s_total;
    const int tid = threadIdx.x;
    if (tid < units) s_n[tid] = ws.n_cand[u0 + tid];
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
        for (int u = 0; u < units; ++u) tot += s_n[u];
        s_total = tot < k ? tot : k;
    }
    if (tid < H) {
        double m = 0.0;
        long long c = 0;
        for (int u = 0; u < units; ++u) {
            m += ws.mass[(u0 + u) * kExplainMaxHops + tid];
            c += ws.count[(u0 + u) * kExplainMaxHops + tid];
        }
        mass[pair * H + tid] = (float)m;
        count[pair * H + tid] = c;
    }
    __syncthreads();
    const int64_t s = src[pair], t = dst[pair];
    for (int e = tid; e < units * k; e += kExplainThreads) {
        const int u = e / k, i = e % k;
        if (i >= s_n[u]) continue;
        const Cand x = ws.cand[(u0 + u) * k + i];
        int rank = i;
        for (int v = 0; v < units && rank < k; ++v) {
            if (v == u) continue;
            const Cand* list = ws.cand + (u0 + v) * k;
            int lo = 0, n = s_n[v];
            while (n > 0) {
                const int half = n >> 1;
                if (beats(list[lo + half], x)) { lo += half + 1; n -= half + 1; } else { n = half; }
            }
            rank += lo;
        }
        if (rank >= k) continue;
        const int64_t o = pair * k + rank;
        hops[o] = x.h;
        weight[o] = x.w;
        int64_t* nd = nodes + o * (H + 1);
        int64_t* sl = slots + o * H;
        nd[0] = s;
        if (x.h == 1) { nd[1] = t; }
        else if (x.h == 2) { nd[1] = x.v1; nd[2] = t; }
        else { nd[1] = x.v1; nd[2] = x.v2; nd[3] = t; }
        for (int m = x.h + 1; m <= H; ++m) nd[m] = -1;
        for (int m = 0; m < H; ++m) sl[m] = m < x.h ? x.slot[m] : -1;
    }
    for (int r = s_total + tid; r < k; r += kExplainThreads) {  // missing paths
        const int64_t o = pair * k + r;
        hops[o] = 0;
        weight[o] = 0.f;
        for (int m = 0; m <= H; ++m) nodes[o * (H + 1) + m] = -1;
        for (int m = 0; m < H; ++m) slots[o * H + m] = -1;
    }
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int64_t kgat_explain_paths_workspace_bytes(int64_t n_pairs, int32_t k, int32_t max_hops) {
    if (n_pairs < 0 || k < 1 || k > kExplainMaxK || max_hops < 1 || max_hops > kExplainMaxHops) return -1;
    return workspace_bytes(n_pairs * explain_units(n_pairs), k);
}

int kgat_explain_paths(const int32_t* row_ptr, const int32_t* col_idx, const float* vals, const int32_t* t_ptr, const int32_t* t_idx,
                       const int32_t* t_perm, int64_t n_nodes, const int32_t* src, const int32_t* dst, int64_t n_pairs, int32_t k,
                       int32_t max_hops, int64_t* nodes, int64_t* slots, int32_t* hops, float* weight, int64_t* count, float* mass,
                       void* workspace, int64_t workspace_bytes_, void* stream) {
    if (n_pairs < 0 || k < 1 || k > kExplainMaxK || max_hops < 1 || max_hops > kExplainMaxHops || n_nodes < 0 || n_nodes > 0x7fffffff)
        return KGAT_ERR_INVALID_ARGUMENT;
    if (n_pairs == 0) return KGAT_OK;
    if (!row_ptr || !col_idx || !vals || !t_ptr || !t_idx || !t_perm || !src || !dst || !nodes || !slots || !hops || !weight || !count ||
        !mass || !workspace)
        return KGAT_ERR_INVALID_ARGUMENT;
    const int units = explain_units(n_pairs);
    const int64_t n_units = n_pairs * units;
    if (workspace_bytes_ < workspace_bytes(n_units, k)) return KGAT_ERR_WORKSPACE;
    if (n_units > 0x7fffffff) return KGAT_ERR_INVALID_ARGUMENT;
    const Workspace ws = carve(workspace, n_units, k);
    const Graph g{row_ptr, col_idx, vals, t_ptr, t_idx, t_perm, n_nodes};
    explain_units_kernel<<<(unsigned)n_units, kExplainThreads, 0, (cudaStream_t)stream>>>(g, src, dst, units, k, max_hops, ws);
    int rc = check_launch();
    if (rc != KGAT_OK) return rc;
    explain_merge_kernel<<<(unsigned)n_pairs, kExplainThreads, 0, (cudaStream_t)stream>>>(src, dst, units, k, max_hops, ws, nodes, slots, hops,
                                                                                          weight, count, mass);
    return check_launch();
}

}  // extern "C"
