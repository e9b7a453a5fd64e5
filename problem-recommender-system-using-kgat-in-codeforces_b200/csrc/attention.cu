// K6-K8: attention refresh on device (reference model.py:263-366, multi_head_attention.py:35-58).
//
// What the reference computes per edge (h, r, t), once the dead query/key path is removed (the
// softmax runs over a length-1 axis and is identically 1, SURVEY.md Q1):
//     x = e_t W_r ;  v = Wv x + bv ;  (per-head dropout on v, train mode only, Q2)
//     o = Wo v + bo ;  y = LayerNorm(o) ;  score = sum_j tanh(y_j)
//     score *= 1 / (log1p(deg_r(h)) + log1p(indeg_r(t)))        (degrees inside the relation batch)
// followed by COO coalescing (duplicate (h, t) summed) and a row softmax on the CPU (Q3).
//
// Here: x, v (and in eval mode the whole score) depend only on the (t, r) pair, so they are computed
// once per UNIQUE pair (pairs arrive sorted by relation: W_r stays in L1/L2); the per-edge work is a
// gather (eval) or one Wo mat-vec (train, because the dropout mask is per edge); the duplicate merge
// and the softmax are one warp-per-row pass over CSR slots -- no host round trip.
#include "common.cuh"

namespace kgat {
namespace {

struct Mha {
    const float* Wv;
    const float* bv;
    const float* Wo;
    const float* bo;
    const float* gamma;
    const float* beta;
    float eps;
    int n_heads;
};

// y = M x + b with M given transposed in shared memory (MT[k][c]); lane owns c = lane + 32 m
template <int DM>
__device__ __forceinline__ void matvec_smem(const float* __restrict__ MT, const float* __restrict__ bias, const float (&x)[DM],
                                            int lane, float (&y)[DM]) {
    constexpr int D = DM * 32;
#pragma unroll
    for (int m = 0; m < DM; ++m) y[m] = bias[lane + 32 * m];
#pragma unroll
    for (int km = 0; km < DM; ++km) {
#pragma unroll 8
        for (int kk = 0; kk < 32; ++kk) {
            const float xv = __shfl_sync(kFull, x[km], kk);
            const float* row = MT + (km * 32 + kk) * D + lane;
#pragma unroll
            for (int m = 0; m < DM; ++m) y[m] = fmaf(xv, row[32 * m], y[m]);
        }
    }
}

// sum_j tanh(LayerNorm(o)_j)
template <int DM>
__device__ __forceinline__ float ln_tanh_sum(const float (&o)[DM], const Mha& P, int lane) {
    constexpr int D = DM * 32;
    float s = 0.f;
#pragma unroll
    for (int m = 0; m < DM; ++m) s += o[m];
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int m = 0; m < DM; ++m) {
        const float c = o[m] - mean;
        q = fmaf(c, c, q);
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)D + P.eps);
    float t = 0.f;
#pragma unroll
    for (int m = 0; m < DM; ++m) t += tanhf((o[m] - mean) * rstd * P.gamma[lane + 32 * m] + P.beta[lane + 32 * m]);
    return warp_sum(t);
}

template <int DM>
__device__ __forceinline__ void stage_transposed(const float* __restrict__ M, float* __restrict__ MT, int tid, int nthreads) {
    constexpr int D = DM * 32;
    for (int i = tid; i < D * D; i += nthreads) {
        const int c = i / D, k = i % D;  // nn.Linear weight [out c][in k]
        MT[k * D + c] = M[i];
    }
}

template <int DM>
__global__ void __launch_bounds__(128) pair_scores_kernel(const float* __restrict__ emb, const float* __restrict__ W,
                                                          const int32_t* __restrict__ pair_tail, const int32_t* __restrict__ pair_rel,
                                                          int64_t n_pairs, Mha P, float* __restrict__ v_out,
                                                          float* __restrict__ score_out) {
    constexpr int D = DM * 32;
    extern __shared__ __align__(16) float smem[];
    float* WvT = smem;
    float* WoT = smem + D * D;
    stage_transposed<DM>(P.Wv, WvT, threadIdx.x, blockDim.x);
    if (score_out != nullptr) stage_transposed<DM>(P.Wo, WoT, threadIdx.x, blockDim.x);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t pr = warp0; pr < n_pairs; pr += nwarps) {
        const int64_t t = pair_tail[pr], r = pair_rel[pr];
        float e[DM], x[DM], v[DM];
#pragma unroll
        for (int m = 0; m < DM; ++m) {
            e[m] = __ldg(emb + t * D + lane + 32 * m);
            x[m] = 0.f;
        }
        const float* Wr = W + r * (int64_t)D * D;
#pragma unroll
        for (int jm = 0; jm < DM; ++jm) {
#pragma unroll 8
            for (int jj = 0; jj < 32; ++jj) {
                const float a = __shfl_sync(kFull, e[jm], jj);
                const float* wrow = Wr + (jm * 32 + jj) * D + lane;
#pragma unroll
                for (int m = 0; m < DM; ++m) x[m] = fmaf(a, __ldg(wrow + 32 * m), x[m]);
            }
        }
        matvec_smem<DM>(WvT, P.bv, x, lane, v);
        if (v_out != nullptr) {
#pragma unroll
            for (int m = 0; m < DM; ++m) v_out[pr * D + lane + 32 * m] = v[m];
        }
        if (score_out != nullptr) {
            float o[DM];
            matvec_smem<DM>(WoT, P.bo, v, lane, o);
            const float s = ln_tanh_sum<DM>(o, P, lane);
            if (lane == 0) score_out[pr] = s;
        }
    }
}

template <int DM>
__global__ void __launch_bounds__(128) edge_scores_dropout_kernel(const float* __restrict__ pair_v,
                                                                  const int32_t* __restrict__ pair_of_edge, int64_t n_edges, Mha P,
                                                                  float dropout_p, const uint8_t* __restrict__ head_bits,
                                                                  uint64_t seed, uint64_t offset,
                                                                  const uint64_t* __restrict__ seed_dev,
                                                                  float* __restrict__ score_out) {
    constexpr int D = DM * 32;
    extern __shared__ __align__(16) float smem[];
    if (seed_dev != nullptr) seed += seed_dev[0] * 0x9E3779B97F4A7C15ull;
    float* WoT = smem;
    stage_transposed<DM>(P.Wo, WoT, threadIdx.x, blockDim.x);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int depth = D / P.n_heads;
    const float scale = 1.f / (1.f - dropout_p);
    const float q = 1.f - dropout_p;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e = warp0; e < n_edges; e += nwarps) {
        uint32_t keep;
        if (head_bits != nullptr) {
            keep = head_bits[e];
        } else {
            const uint4 rnd = philox4x32(seed, offset + (uint64_t)e);
            const uint32_t w[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
            keep = 0;
            for (int hd = 0; hd < P.n_heads && hd < 8; ++hd) {
                const uint32_t bits16 = (w[hd >> 1] >> ((hd & 1) * 16)) & 0xffffu;
                if ((float)bits16 * (1.f / 65536.f) < q) keep |= 1u << hd;
            }
        }
        const int64_t pr = pair_of_edge[e];
        float v[DM], o[DM];
#pragma unroll
        for (int m = 0; m < DM; ++m) {
            const int c = lane + 32 * m;
            const float val = __ldg(pair_v + pr * D + c);
            v[m] = ((keep >> (c / depth)) & 1u) ? val * scale : 0.f;
        }
        matvec_smem<DM>(WoT, P.bo, v, lane, o);
        const float s = ln_tanh_sum<DM>(o, P, lane);
        if (lane == 0) score_out[e] = s;
    }
}

// MultiHeadAttention.forward on caller-provided (already projected) tail embeddings (multi_head_attention.py:35-58):
// y = LayerNorm(Wo drop(Wv x + bv) + bo).  The query / key inputs do not influence the output (softmax over a
// length-1 axis), so only x = tail_embedding is read.  One warp per row.
template <int DM>
__global__ void __launch_bounds__(128) mha_forward_kernel(const float* __restrict__ x_in, int64_t n, Mha P, float dropout_p,
                                                          const uint8_t* __restrict__ head_bits, uint64_t seed, uint64_t offset,
                                                          float* __restrict__ y_out) {
    constexpr int D = DM * 32;
    extern __shared__ __align__(16) float smem[];
    float* WvT = smem;
    float* WoT = smem + D * D;
    stage_transposed<DM>(P.Wv, WvT, threadIdx.x, blockDim.x);
    stage_transposed<DM>(P.Wo, WoT, threadIdx.x, blockDim.x);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int depth = D / P.n_heads;
    const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    const float q = 1.f - dropout_p;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp0; i < n; i += nwarps) {
        float x[DM], v[DM], o[DM];
#pragma unroll
        for (int m = 0; m < DM; ++m) x[m] = __ldg(x_in + i * D + lane + 32 * m);
        matvec_smem<DM>(WvT, P.bv, x, lane, v);
        if (dropout_p > 0.f) {
            uint32_t keep;
            if (head_bits != nullptr) {
                keep = head_bits[i];
            } else {
                const uint4 rnd = philox4x32(seed, offset + (uint64_t)i);
                const uint32_t w[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
                keep = 0;
                for (int hd = 0; hd < P.n_heads && hd < 8; ++hd) {
                    const uint32_t bits16 = (w[hd >> 1] >> ((hd & 1) * 16)) & 0xffffu;
                    if ((float)bits16 * (1.f / 65536.f) < q) keep |= 1u << hd;
                }
            }
#pragma unroll
            for (int m = 0; m < DM; ++m) v[m] = ((keep >> ((lane + 32 * m) / depth)) & 1u) ? v[m] * scale : 0.f;
        }
        matvec_smem<DM>(WoT, P.bo, v, lane, o);
        float s = 0.f;
#pragma unroll
        for (int m = 0; m < DM; ++m) s += o[m];
        const float mean = warp_sum(s) / (float)D;
        float qq = 0.f;
#pragma unroll
        for (int m = 0; m < DM; ++m) {
            const float c = o[m] - mean;
            qq = fmaf(c, c, qq);
        }
        const float rstd = rsqrtf(warp_sum(qq) / (float)D + P.eps);
#pragma unroll
        for (int m = 0; m < DM; ++m)
            y_out[i * D + lane + 32 * m] = (o[m] - mean) * rstd * P.gamma[lane + 32 * m] + P.beta[lane + 32 * m];
    }
}

// Canonical KGAT attention score (north_star item (1), the paper's pi(h, r, t) = (W_r e_t)^T tanh(W_r e_h + e_r), in the
// reference's row-vector convention x = e W_r, model.py:291-298) -- NOT what the reference computes (SURVEY.md Q1); offered as
// model.score_mode = "kgat".  Step 1: x = e W_r once per unique (node, relation) pair; step 2: one warp per edge gathers its
// two projections and e_r.
template <int DM>
__global__ void __launch_bounds__(128) pair_project_kernel(const float* __restrict__ emb, const float* __restrict__ W,
                                                           const int32_t* __restrict__ pair_node, const int32_t* __restrict__ pair_rel,
                                                           int64_t n_pairs, float* __restrict__ x_out) {
    constexpr int D = DM * 32;
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t pr = warp0; pr < n_pairs; pr += nwarps) {
        const int64_t t = pair_node[pr], r = pair_rel[pr];
        float e[DM], x[DM];
#pragma unroll
        for (int m = 0; m < DM; ++m) {
            e[m] = __ldg(emb + t * D + lane + 32 * m);
            x[m] = 0.f;
        }
        const float* Wr = W + r * (int64_t)D * D;
#pragma unroll
        for (int jm = 0; jm < DM; ++jm) {
#pragma unroll 8
            for (int jj = 0; jj < 32; ++jj) {
                const float a = __shfl_sync(kFull, e[jm], jj);
                const float* wrow = Wr + (jm * 32 + jj) * D + lane;
#pragma unroll
                for (int m = 0; m < DM; ++m) x[m] = fmaf(a, __ldg(wrow + 32 * m), x[m]);
            }
        }
#pragma unroll
        for (int m = 0; m < DM; ++m) x_out[pr * D + lane + 32 * m] = x[m];
    }
}

__global__ void __launch_bounds__(128) edge_scores_kgat_kernel(const float* __restrict__ x_head, const int32_t* __restrict__ head_pair,
                                                               const float* __restrict__ x_tail, const int32_t* __restrict__ tail_pair,
                                                               const float* __restrict__ rel_emb, const int32_t* __restrict__ edge_rel,
                                                               int64_t n_edges, int d, float* __restrict__ score_out) {
    const int lane = threadIdx.x & 31;
    const int64_t e = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (e >= n_edges) return;
    const float* xh = x_head + (int64_t)head_pair[e] * d;
    const float* xt = x_tail + (int64_t)tail_pair[e] * d;
    const float* er = rel_emb + (int64_t)edge_rel[e] * d;
    float s = 0.f;
    for (int j = lane; j < d; j += 32) s = fmaf(__ldg(xt + j), tanhf(__ldg(xh + j) + __ldg(er + j)), s);
    s = warp_sum(s);
    if (lane == 0) score_out[e] = s;
}

__global__ void __launch_bounds__(128) row_softmax_kernel(const int32_t* __restrict__ row_ptr, int64_t n_rows,
                                                          const int32_t* __restrict__ slot_ptr, const float* __restrict__ pair_score,
                                                          const int32_t* __restrict__ pair_of_edge,
                                                          const float* __restrict__ edge_score,
                                                          const float* __restrict__ edge_weight, float* __restrict__ vals) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (row >= n_rows) return;
    const int b = row_ptr[row], e = row_ptr[row + 1];
    if (b == e) return;
    float mx = -INFINITY;
    for (int s = b + lane; s < e; s += 32) {
        const int pb = slot_ptr[s], pe = slot_ptr[s + 1];
        float acc = 0.f;
        for (int p = pb; p < pe; ++p) {
            const float sc = pair_score != nullptr ? pair_score[pair_of_edge[p]] : edge_score[p];
            const float term = sc * edge_weight[p];
            acc = (p == pb) ? term : acc + term;
        }
        vals[s] = acc;
        mx = fmaxf(mx, acc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int s = b + lane; s < e; s += 32) {
        const float ex = expf(vals[s] - mx);
        vals[s] = ex;
        sum += ex;
    }
    sum = warp_sum(sum);
    for (int s = b + lane; s < e; s += 32) vals[s] = vals[s] / sum;
}

__global__ void edge_weights_kernel(const int32_t* __restrict__ dh, const int32_t* __restrict__ dt, const float* __restrict__ mult,
                                    int64_t n, float* __restrict__ w) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v = 1.0f / (log1pf((float)dh[i]) + log1pf((float)dt[i]));
    if (mult != nullptr) v *= mult[i];
    w[i] = v;
}

int pack_mha(const kgat_mha_t* m, Mha* out) {
    if (!m || !m->Wv || !m->bv || !m->Wo || !m->bo || !m->ln_gamma || !m->ln_beta || m->n_heads <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    *out = Mha{m->Wv, m->bv, m->Wo, m->bo, m->ln_gamma, m->ln_beta, m->ln_eps, m->n_heads};
    return KGAT_OK;
}

template <int DM>
int launch_pairs(const float* emb, const float* W, const int32_t* pt, const int32_t* pr, int64_t n_pairs, const Mha& P, float* v_out,
                 float* score_out, cudaStream_t stream) {
    constexpr int D = DM * 32;
    const size_t smem = sizeof(float) * 2 * D * D;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(pair_scores_kernel<DM>, (int)smem, configured); rc != KGAT_OK) return rc;
    int64_t blocks = (n_pairs + 3) / 4;
    const int64_t cap = (int64_t)sm_count() * (DM <= 2 ? 4 : 1);
    if (blocks > cap) blocks = cap;
    pair_scores_kernel<DM><<<(unsigned)blocks, 128, smem, stream>>>(emb, W, pt, pr, n_pairs, P, v_out, score_out);
    return check_launch();
}

template <int DM>
int launch_edges(const float* pair_v, const int32_t* poe, int64_t n_edges, const Mha& P, float p, const uint8_t* head_bits, uint64_t seed,
                 uint64_t offset, const uint64_t* seed_dev, float* score_out, cudaStream_t stream) {
    constexpr int D = DM * 32;
    const size_t smem = sizeof(float) * D * D;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(edge_scores_dropout_kernel<DM>, (int)smem, configured); rc != KGAT_OK) return rc;
    int64_t blocks = (n_edges + 3) / 4;
    const int64_t cap = (int64_t)sm_count() * (DM <= 2 ? 8 : 2);
    if (blocks > cap) blocks = cap;
    edge_scores_dropout_kernel<DM><<<(unsigned)blocks, 128, smem, stream>>>(pair_v, poe, n_edges, P, p, head_bits, seed, offset, seed_dev,
                                                                            score_out);
    return check_launch();
}

template <int DM>
int launch_mha(const float* x, int64_t n, const Mha& P, float p, const uint8_t* head_bits, uint64_t seed, uint64_t offset, float* y,
               cudaStream_t stream) {
    constexpr int D = DM * 32;
    const size_t smem = sizeof(float) * 2 * D * D;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(mha_forward_kernel<DM>, (int)smem, configured); rc != KGAT_OK) return rc;
    int64_t blocks = (n + 3) / 4;
    const int64_t cap = (int64_t)sm_count() * (DM <= 2 ? 4 : 1);
    if (blocks > cap) blocks = cap;
    mha_forward_kernel<DM><<<(unsigned)blocks, 128, smem, stream>>>(x, n, P, p, head_bits, seed, offset, y);
    return check_launch();
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int kgat_mha_forward(const float* tail_embedding, int64_t n, int32_t d, const kgat_mha_t* mha, float dropout_p, const uint8_t* head_bits,
                     uint64_t seed, uint64_t offset, float* out, void* stream) {
    Mha P;
    int rc = pack_mha(mha, &P);
    if (rc != KGAT_OK) return rc;
    if (n < 0 || dropout_p < 0.f || dropout_p >= 1.f || P.n_heads > 8 || d % P.n_heads) return KGAT_ERR_INVALID_ARGUMENT;
    if (n == 0) return KGAT_OK;
    switch (d) {
        case 32: return launch_mha<1>(tail_embedding, n, P, dropout_p, head_bits, seed, offset, out, (cudaStream_t)stream);
        case 64: return launch_mha<2>(tail_embedding, n, P, dropout_p, head_bits, seed, offset, out, (cudaStream_t)stream);
        case 128: return launch_mha<4>(tail_embedding, n, P, dropout_p, head_bits, seed, offset, out, (cudaStream_t)stream);
        default: return KGAT_ERR_UNSUPPORTED;
    }
}

int kgat_att_pair_project(const float* emb, const float* W, int32_t d, const int32_t* pair_node, const int32_t* pair_rel, int64_t n_pairs,
                          float* x_out, void* stream) {
    if (!emb || !W || !pair_node || !pair_rel || !x_out || n_pairs < 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_pairs == 0) return KGAT_OK;
    int64_t blocks = (n_pairs + 3) / 4;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    switch (d) {
        case 32: pair_project_kernel<1><<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(emb, W, pair_node, pair_rel, n_pairs, x_out); break;
        case 64: pair_project_kernel<2><<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(emb, W, pair_node, pair_rel, n_pairs, x_out); break;
        case 128: pair_project_kernel<4><<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(emb, W, pair_node, pair_rel, n_pairs, x_out); break;
        default: return KGAT_ERR_UNSUPPORTED;
    }
    return check_launch();
}

int kgat_att_edge_scores_kgat(const float* x_head, const int32_t* head_pair, const float* x_tail, const int32_t* tail_pair, const float* rel_emb,
                              const int32_t* edge_rel, int64_t n_edges, int32_t d, float* score_out, void* stream) {
    if (!x_head || !head_pair || !x_tail || !tail_pair || !rel_emb || !edge_rel || !score_out || n_edges < 0 || d <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_edges == 0) return KGAT_OK;
    const unsigned blocks = (unsigned)((n_edges * 32 + 127) / 128);
    edge_scores_kgat_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(x_head, head_pair, x_tail, tail_pair, rel_emb, edge_rel, n_edges, d, score_out);
    return check_launch();
}

int kgat_att_pair_scores(const float* emb, const float* W, int32_t d, const int32_t* pair_tail, const int32_t* pair_rel, int64_t n_pairs,
                         const kgat_mha_t* mha, float* v_out, float* score_out, void* stream) {
    Mha P;
    int rc = pack_mha(mha, &P);
    if (rc != KGAT_OK) return rc;
    if (n_pairs < 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_pairs == 0) return KGAT_OK;
    switch (d) {
        case 32: return launch_pairs<1>(emb, W, pair_tail, pair_rel, n_pairs, P, v_out, score_out, (cudaStream_t)stream);
        case 64: return launch_pairs<2>(emb, W, pair_tail, pair_rel, n_pairs, P, v_out, score_out, (cudaStream_t)stream);
        case 128: return launch_pairs<4>(emb, W, pair_tail, pair_rel, n_pairs, P, v_out, score_out, (cudaStream_t)stream);
        default: return KGAT_ERR_UNSUPPORTED;
    }
}

int kgat_att_edge_scores_dropout(const float* pair_v, const int32_t* pair_of_edge, int64_t n_edges, int32_t d, const kgat_mha_t* mha,
                                 float dropout_p, const uint8_t* head_bits, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                                 float* score_out, void* stream) {
    Mha P;
    int rc = pack_mha(mha, &P);
    if (rc != KGAT_OK) return rc;
    if (n_edges < 0 || dropout_p < 0.f || dropout_p >= 1.f || P.n_heads > 8 || d % P.n_heads) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_edges == 0) return KGAT_OK;
    switch (d) {
        case 32: return launch_edges<1>(pair_v, pair_of_edge, n_edges, P, dropout_p, head_bits, seed, offset, seed_dev, score_out, (cudaStream_t)stream);
        case 64: return launch_edges<2>(pair_v, pair_of_edge, n_edges, P, dropout_p, head_bits, seed, offset, seed_dev, score_out, (cudaStream_t)stream);
        case 128: return launch_edges<4>(pair_v, pair_of_edge, n_edges, P, dropout_p, head_bits, seed, offset, seed_dev, score_out, (cudaStream_t)stream);
        default: return KGAT_ERR_UNSUPPORTED;
    }
}

int kgat_att_row_softmax(const int32_t* row_ptr, int64_t n_rows, const int32_t* slot_ptr, const float* pair_score,
                         const int32_t* pair_of_edge, const float* edge_score, const float* edge_weight, float* vals, void* stream) {
    if (n_rows < 0 || (!pair_score && !edge_score) || (pair_score && !pair_of_edge)) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_rows == 0) return KGAT_OK;
    const unsigned blocks = (unsigned)((n_rows * 32 + 127) / 128);
    row_softmax_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(row_ptr, n_rows, slot_ptr, pair_score, pair_of_edge, edge_score,
                                                                edge_weight, vals);
    return check_launch();
}

int kgat_att_edge_weights(const int32_t* deg_head, const int32_t* deg_tail, const float* mult, int64_t n_edges, float* edge_weight,
                          void* stream) {
    if (n_edges < 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_edges == 0) return KGAT_OK;
    edge_weights_kernel<<<(unsigned)((n_edges + 255) / 256), 256, 0, (cudaStream_t)stream>>>(deg_head, deg_tail, mult, n_edges, edge_weight);
    return check_launch();
}

}  // extern "C"
