// K2/K3: fused bi-interaction aggregator, forward and hand-written backward.
// Replaces, per propagation layer, two nn.Linear GEMMs + LeakyReLU x2 + add + Dropout + F.normalize
// (reference aggregator.py:57-65) and their autograd backward with ONE kernel each way.
//
//   forward : out = normalize( drop( lrelu((E+S) W1^T + b1) + lrelu((E*S) W2^T + b2) ) )
//   backward: g_S, g_E(direct), and per-CTA partial dW1, db1, dW2, db2 (reduced in fixed order)
//
// Tiling: a CTA owns TM rows; (E+S) / (E*S) tiles and both weight matrices live in shared memory,
// every thread keeps an RM x 4 register micro-tile per product, rows are normalised with a
// shuffle reduction over the DOUT/4 threads that share a row.  The CTAs are persistent (grid =
// k x #SM) so weights are staged once and weight-gradient accumulators stay in registers across
// row tiles.  fp32 FMA throughout: results stay inside the 1e-5 parity budget.
#include <stdlib.h>

#include "common.cuh"

namespace kgat {
namespace {

template <int DIN, int DOUT>
struct Cfg {
    static constexpr bool kBig = (DIN > 64) || (DOUT > 64);
    static constexpr int TM = kBig ? 32 : 64;    // rows per tile
    static constexpr int NT = kBig ? 512 : 256;  // threads per CTA
    static constexpr int SE = DIN + 4;           // smem row stride of input tiles
    static constexpr int SG = DOUT + 4;          // smem row stride of gz tiles
    // forward / phase-1 mapping over the TM x DOUT tile
    static constexpr int CG = DOUT / 4;          // threads per row
    static constexpr int RGROUPS = NT / CG;
    static constexpr int RM = TM / RGROUPS;      // rows per thread
    // backward phase-2 mapping over the TM x DIN tile
    static constexpr int KG = DIN / 4;
    static constexpr int RGROUPS2 = NT / KG;
    static constexpr int RM2 = TM / RGROUPS2;
    // backward phase-3 mapping over the DOUT x DIN weight tile
    static constexpr int CROWS = (NT / KG) < DOUT ? (NT / KG) : DOUT;
    static constexpr int CPT = DOUT / CROWS;
    static constexpr int ACTIVE3 = CROWS * KG;
    static_assert(RM >= 1 && RM * RGROUPS == TM, "bad forward mapping");
    static_assert(RM2 >= 1 && RM2 * RGROUPS2 == TM, "bad phase-2 mapping");
    static_assert(CPT >= 1 && CPT * CROWS == DOUT, "bad phase-3 mapping");
    static constexpr size_t fwd_smem = sizeof(float) * (2 * DIN * DOUT + 2 * TM * SE);
    static constexpr size_t bwd_smem = sizeof(float) * (2 * DIN * DOUT + 2 * TM * SE + 2 * TM * SG);
};

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <int DIN, int DOUT>
__global__ void __launch_bounds__(Cfg<DIN, DOUT>::NT) biagg_fwd_kernel(
    const float* __restrict__ E, const float* __restrict__ S, int64_t n, const float* __restrict__ W1,
    const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2, float dropout_p,
    uint64_t seed, uint64_t offset, const uint64_t* __restrict__ seed_dev, const uint32_t* __restrict__ keep_bits,
    float* __restrict__ out, int64_t ld_out, float* __restrict__ inv_norm, uint8_t* __restrict__ flags) {
    using C = Cfg<DIN, DOUT>;
    extern __shared__ __align__(16) float smem[];
    if (seed_dev != nullptr) seed += seed_dev[0] * 0x9E3779B97F4A7C15ull;  // per-step stream under CUDA-graph replay
    float* W1t = smem;                  // [DIN][DOUT]  (transposed nn.Linear weight)
    float* W2t = W1t + DIN * DOUT;      // [DIN][DOUT]
    float* Us = W2t + DIN * DOUT;       // [TM][SE]   E + S
    float* Vs = Us + C::TM * C::SE;     // [TM][SE]   E * S
    const int tid = threadIdx.x;

    for (int i = tid; i < DIN * DOUT; i += C::NT) {
        const int c = i / DIN, k = i % DIN;  // W[c][k] coalesced read
        W1t[k * DOUT + c] = W1[i];
        W2t[k * DOUT + c] = W2[i];
    }
    const int cg = tid % C::CG, rg = tid / C::CG;
    float bias1[4], bias2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        bias1[j] = b1[cg * 4 + j];
        bias2[j] = b2[cg * 4 + j];
    }
    const float keep_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    const int words_per_row = (DOUT + 31) / 32;
    const int64_t n_tiles = (n + C::TM - 1) / C::TM;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * C::TM;
        __syncthreads();  // previous tile fully consumed (also orders the weight staging)
        for (int i = tid; i < C::TM * (DIN / 4); i += C::NT) {
            const int r = i / (DIN / 4), q = i % (DIN / 4);
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f), s = e;
            if (row0 + r < n) {
                e = ld_stream4(E + (row0 + r) * DIN + q * 4);
                s = ld_stream4(S + (row0 + r) * DIN + q * 4);
            }
            *reinterpret_cast<float4*>(Us + r * C::SE + q * 4) = make_float4(e.x + s.x, e.y + s.y, e.z + s.z, e.w + s.w);
            *reinterpret_cast<float4*>(Vs + r * C::SE + q * 4) = make_float4(e.x * s.x, e.y * s.y, e.z * s.z, e.w * s.w);
        }
        __syncthreads();

        float z1[C::RM][4], z2[C::RM][4];
#pragma unroll
        for (int i = 0; i < C::RM; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                z1[i][j] = bias1[j];
                z2[i][j] = bias2[j];
            }
#pragma unroll 2
        for (int k4 = 0; k4 < DIN / 4; ++k4) {
            float4 u[C::RM], v[C::RM];
#pragma unroll
            for (int i = 0; i < C::RM; ++i) {
                const int r = rg * C::RM + i;
                u[i] = *reinterpret_cast<const float4*>(Us + r * C::SE + k4 * 4);
                v[i] = *reinterpret_cast<const float4*>(Vs + r * C::SE + k4 * 4);
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float4 w1 = *reinterpret_cast<const float4*>(W1t + (k4 * 4 + kk) * DOUT + cg * 4);
                const float4 w2 = *reinterpret_cast<const float4*>(W2t + (k4 * 4 + kk) * DOUT + cg * 4);
#pragma unroll
                for (int i = 0; i < C::RM; ++i) {
                    const float uu = kk == 0 ? u[i].x : kk == 1 ? u[i].y : kk == 2 ? u[i].z : u[i].w;
                    const float vv = kk == 0 ? v[i].x : kk == 1 ? v[i].y : kk == 2 ? v[i].z : v[i].w;
                    z1[i][0] = fmaf(uu, w1.x, z1[i][0]);
                    z1[i][1] = fmaf(uu, w1.y, z1[i][1]);
                    z1[i][2] = fmaf(uu, w1.z, z1[i][2]);
                    z1[i][3] = fmaf(uu, w1.w, z1[i][3]);
                    z2[i][0] = fmaf(vv, w2.x, z2[i][0]);
                    z2[i][1] = fmaf(vv, w2.y, z2[i][1]);
                    z2[i][2] = fmaf(vv, w2.z, z2[i][2]);
                    z2[i][3] = fmaf(vv, w2.w, z2[i][3]);
                }
            }
        }

        // epilogue: activation, dropout, row L2 normalisation
#pragma unroll
        for (int i = 0; i < C::RM; ++i) {
            const int64_t row = row0 + rg * C::RM + i;
            const bool valid = row < n;
            uint32_t keep = 0xfu;
            if (dropout_p > 0.f && valid) {
                if (keep_bits != nullptr) {
                    const uint32_t wbits = keep_bits[row * words_per_row + (cg * 4) / 32];
                    keep = (wbits >> ((cg * 4) & 31)) & 0xfu;
                } else {
                    const uint4 rnd = philox4x32(seed, offset + (uint64_t)row * C::CG + cg);
                    const float q = 1.f - dropout_p;
                    keep = (u01(rnd.x) < q ? 1u : 0u) | (u01(rnd.y) < q ? 2u : 0u) | (u01(rnd.z) < q ? 4u : 0u) |
                           (u01(rnd.w) < q ? 8u : 0u);
                }
            }
            float x[4];
            uint8_t f[4];
            float ss = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const bool kp = (keep >> j) & 1u;
                f[j] = (z1[i][j] > 0.f ? 1 : 0) | (z2[i][j] > 0.f ? 2 : 0) | (kp ? 4 : 0);
                const float a = lrelu(z1[i][j]) + lrelu(z2[i][j]);
                x[j] = kp ? a * keep_scale : 0.f;
                ss = fmaf(x[j], x[j], ss);
            }
#pragma unroll
            for (int o = 1; o < C::CG; o <<= 1) ss += __shfl_xor_sync(kFull, ss, o);
            const float nrm = sqrtf(ss);
            const float denom = fmaxf(nrm, KGAT_NORM_EPS);
            if (valid) {
                *reinterpret_cast<float4*>(out + row * ld_out + cg * 4) =
                    make_float4(x[0] / denom, x[1] / denom, x[2] / denom, x[3] / denom);
                if (flags != nullptr) *reinterpret_cast<uchar4*>(flags + row * DOUT + cg * 4) = make_uchar4(f[0], f[1], f[2], f[3]);
                if (inv_norm != nullptr && cg == 0) inv_norm[row] = nrm < KGAT_NORM_EPS ? -1.f / denom : 1.f / denom;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
template <int DIN, int DOUT>
__global__ void __launch_bounds__(Cfg<DIN, DOUT>::NT) biagg_bwd_kernel(
    const float* __restrict__ g_out, int64_t ld_gout, const float* __restrict__ out, int64_t ld_out,
    const float* __restrict__ inv_norm, const uint8_t* __restrict__ flags, const float* __restrict__ E,
    const float* __restrict__ S, int64_t n, const float* __restrict__ W1, const float* __restrict__ W2, float dropout_p,
    float* __restrict__ g_S, float* __restrict__ g_E, float* __restrict__ partials) {
    using C = Cfg<DIN, DOUT>;
    extern __shared__ __align__(16) float smem[];
    float* W1s = smem;                   // [DOUT][DIN] as stored
    float* W2s = W1s + DIN * DOUT;
    float* Es = W2s + DIN * DOUT;        // [TM][SE]
    float* Ss = Es + C::TM * C::SE;      // [TM][SE]
    float* G1 = Ss + C::TM * C::SE;      // [TM][SG]  dL/dz1
    float* G2 = G1 + C::TM * C::SG;      // [TM][SG]  dL/dz2
    const int tid = threadIdx.x;

    for (int i = tid; i < DIN * DOUT / 4; i += C::NT) {
        reinterpret_cast<float4*>(W1s)[i] = __ldg(reinterpret_cast<const float4*>(W1) + i);
        reinterpret_cast<float4*>(W2s)[i] = __ldg(reinterpret_cast<const float4*>(W2) + i);
    }
    const float keep_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    const int cg = tid % C::CG, rg = tid / C::CG;      // phase 1
    const int kg = tid % C::KG, rg2 = tid / C::KG;     // phase 2
    const int crow = tid / C::KG;                      // phase 3 (kg shared with phase 2)
    const bool act3 = tid < C::ACTIVE3;

    float aw1[C::CPT][4], aw2[C::CPT][4], ab1[C::CPT], ab2[C::CPT];
#pragma unroll
    for (int ci = 0; ci < C::CPT; ++ci) {
        ab1[ci] = ab2[ci] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) aw1[ci][j] = aw2[ci][j] = 0.f;
    }

    const int64_t n_tiles = (n + C::TM - 1) / C::TM;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * C::TM;
        __syncthreads();
        // ---- stage E, S ----
        for (int i = tid; i < C::TM * (DIN / 4); i += C::NT) {
            const int r = i / (DIN / 4), q = i % (DIN / 4);
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f), s = e;
            if (row0 + r < n) {
                e = ld_stream4(E + (row0 + r) * DIN + q * 4);
                s = ld_stream4(S + (row0 + r) * DIN + q * 4);
            }
            *reinterpret_cast<float4*>(Es + r * C::SE + q * 4) = e;
            *reinterpret_cast<float4*>(Ss + r * C::SE + q * 4) = s;
        }
        // ---- phase 1: normalise / dropout / LeakyReLU backward -> dL/dz1, dL/dz2 ----
#pragma unroll
        for (int i = 0; i < C::RM; ++i) {
            const int r = rg * C::RM + i;
            const int64_t row = row0 + r;
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f), y = g;
            uchar4 f = make_uchar4(0, 0, 0, 0);
            float inv = 0.f;
            if (row < n) {
                g = ld_stream4(g_out + row * ld_gout + cg * 4);
                y = ld_stream4(out + row * ld_out + cg * 4);
                f = *reinterpret_cast<const uchar4*>(flags + row * DOUT + cg * 4);
                inv = inv_norm[row];
            }
            float t = g.x * y.x + g.y * y.y + g.z * y.z + g.w * y.w;
#pragma unroll
            for (int o = 1; o < C::CG; o <<= 1) t += __shfl_xor_sync(kFull, t, o);
            if (inv < 0.f) {  // eps clamp was active: y = x / eps, no projection term
                t = 0.f;
                inv = -inv;
            }
            const float gx[4] = {inv * (g.x - y.x * t), inv * (g.y - y.y * t), inv * (g.z - y.z * t), inv * (g.w - y.w * t)};
            const uint8_t fl[4] = {f.x, f.y, f.z, f.w};
            float a1[4], a2[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float gd = (fl[j] & 4) ? gx[j] * keep_scale : 0.f;
                a1[j] = (fl[j] & 1) ? gd : gd * KGAT_LEAKY_SLOPE;
                a2[j] = (fl[j] & 2) ? gd : gd * KGAT_LEAKY_SLOPE;
            }
            *reinterpret_cast<float4*>(G1 + r * C::SG + cg * 4) = make_float4(a1[0], a1[1], a1[2], a1[3]);
            *reinterpret_cast<float4*>(G2 + r * C::SG + cg * 4) = make_float4(a2[0], a2[1], a2[2], a2[3]);
        }
        __syncthreads();

        // ---- phase 2: input gradients  gu = G1 W1, gv = G2 W2 ----
        {
            float gu[C::RM2][4], gv[C::RM2][4];
#pragma unroll
            for (int i = 0; i < C::RM2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) gu[i][j] = gv[i][j] = 0.f;
#pragma unroll 2
            for (int c4 = 0; c4 < DOUT / 4; ++c4) {
                float4 a[C::RM2], b[C::RM2];
#pragma unroll
                for (int i = 0; i < C::RM2; ++i) {
                    const int r = rg2 * C::RM2 + i;
                    a[i] = *reinterpret_cast<const float4*>(G1 + r * C::SG + c4 * 4);
                    b[i] = *reinterpret_cast<const float4*>(G2 + r * C::SG + c4 * 4);
                }
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const float4 w1 = *reinterpret_cast<const float4*>(W1s + (c4 * 4 + cc) * DIN + kg * 4);
                    const float4 w2 = *reinterpret_cast<const float4*>(W2s + (c4 * 4 + cc) * DIN + kg * 4);
#pragma unroll
                    for (int i = 0; i < C::RM2; ++i) {
                        const float aa = cc == 0 ? a[i].x : cc == 1 ? a[i].y : cc == 2 ? a[i].z : a[i].w;
                        const float bb = cc == 0 ? b[i].x : cc == 1 ? b[i].y : cc == 2 ? b[i].z : b[i].w;
                        gu[i][0] = fmaf(aa, w1.x, gu[i][0]);
                        gu[i][1] = fmaf(aa, w1.y, gu[i][1]);
                        gu[i][2] = fmaf(aa, w1.z, gu[i][2]);
                        gu[i][3] = fmaf(aa, w1.w, gu[i][3]);
                        gv[i][0] = fmaf(bb, w2.x, gv[i][0]);
                        gv[i][1] = fmaf(bb, w2.y, gv[i][1]);
                        gv[i][2] = fmaf(bb, w2.z, gv[i][2]);
                        gv[i][3] = fmaf(bb, w2.w, gv[i][3]);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < C::RM2; ++i) {
                const int r = rg2 * C::RM2 + i;
                const int64_t row = row0 + r;
                if (row < n) {
                    const float4 e = *reinterpret_cast<const float4*>(Es + r * C::SE + kg * 4);
                    const float4 s = *reinterpret_cast<const float4*>(Ss + r * C::SE + kg * 4);
                    // u = E + S, v = E * S:  dS = gu + gv * E,  dE = gu + gv * S
                    *reinterpret_cast<float4*>(g_S + row * DIN + kg * 4) =
                        make_float4(fmaf(gv[i][0], e.x, gu[i][0]), fmaf(gv[i][1], e.y, gu[i][1]), fmaf(gv[i][2], e.z, gu[i][2]),
                                    fmaf(gv[i][3], e.w, gu[i][3]));
                    *reinterpret_cast<float4*>(g_E + row * DIN + kg * 4) =
                        make_float4(fmaf(gv[i][0], s.x, gu[i][0]), fmaf(gv[i][1], s.y, gu[i][1]), fmaf(gv[i][2], s.z, gu[i][2]),
                                    fmaf(gv[i][3], s.w, gu[i][3]));
                }
            }
        }

        // ---- phase 3: weight gradients  dW1 += G1^T (E+S),  dW2 += G2^T (E*S),  db += colsum(G) ----
        if (act3) {
#pragma unroll 4
            for (int r = 0; r < C::TM; ++r) {
                const float4 e = *reinterpret_cast<const float4*>(Es + r * C::SE + kg * 4);
                const float4 s = *reinterpret_cast<const float4*>(Ss + r * C::SE + kg * 4);
                const float u[4] = {e.x + s.x, e.y + s.y, e.z + s.z, e.w + s.w};
                const float v[4] = {e.x * s.x, e.y * s.y, e.z * s.z, e.w * s.w};
#pragma unroll
                for (int ci = 0; ci < C::CPT; ++ci) {
                    const float a = G1[r * C::SG + crow * C::CPT + ci];
                    const float b = G2[r * C::SG + crow * C::CPT + ci];
                    ab1[ci] += a;
                    ab2[ci] += b;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        aw1[ci][j] = fmaf(a, u[j], aw1[ci][j]);
                        aw2[ci][j] = fmaf(b, v[j], aw2[ci][j]);
                    }
                }
            }
        }
    }

    // per-CTA partial parameter gradients: [dW1 (DOUT x DIN)][dW2][db1 (DOUT)][db2]
    if (act3) {
        float* p = partials + (int64_t)blockIdx.x * (2 * DIN * DOUT + 2 * DOUT);
#pragma unroll
        for (int ci = 0; ci < C::CPT; ++ci) {
            const int c = crow * C::CPT + ci;
            *reinterpret_cast<float4*>(p + c * DIN + kg * 4) = make_float4(aw1[ci][0], aw1[ci][1], aw1[ci][2], aw1[ci][3]);
            *reinterpret_cast<float4*>(p + DIN * DOUT + c * DIN + kg * 4) = make_float4(aw2[ci][0], aw2[ci][1], aw2[ci][2], aw2[ci][3]);
            if (kg == 0) {
                p[2 * DIN * DOUT + c] = ab1[ci];
                p[2 * DIN * DOUT + DOUT + c] = ab2[ci];
            }
        }
    }
}

// Sum the per-CTA partial parameter gradients in a fixed order (deterministic).  A block owns 32 output
// elements; its 32 warps each add a strided 32nd of the CTAs (296 persistent CTAs: a chain of <= 10 loads per warp -- with 8 warps
// the 37-deep chains made this a 8-12 us kernel), then the 32 sub-sums are added in warp order.
constexpr int kReduceParts = 32;
__global__ void __launch_bounds__(32 * kReduceParts) reduce_partials_kernel(const float* __restrict__ partials, int n_ctas, int din, int dout,
                                                                           float* __restrict__ gW1, float* __restrict__ gb1,
                                                                           float* __restrict__ gW2, float* __restrict__ gb2, int accumulate) {
    __shared__ float sub[kReduceParts][32];
    const int total = 2 * din * dout + 2 * dout;
    const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;
    float s = 0.f;
    if (i < total)
        for (int c = part; c < n_ctas; c += kReduceParts) s += partials[(int64_t)c * total + i];
    sub[part][lane] = s;
    __syncthreads();
    if (part != 0 || i >= total) return;
#pragma unroll
    for (int q = 1; q < kReduceParts; ++q) s += sub[q][lane];
    float* dst;
    if (i < din * dout) dst = gW1 + i;
    else if (i < 2 * din * dout) dst = gW2 + (i - din * dout);
    else if (i < 2 * din * dout + dout) dst = gb1 + (i - 2 * din * dout);
    else dst = gb2 + (i - 2 * din * dout - dout);
    *dst = accumulate ? *dst + s : s;
}

int grid_for(int64_t n, int tm, size_t smem_bytes) {
    const int64_t tiles = (n + tm - 1) / tm;
    int per_sm = (int)(200 * 1024 / (smem_bytes + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    const int64_t cap = (int64_t)sm_count() * per_sm;
    return (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
}

template <int DIN, int DOUT>
int launch_fwd(const float* E, const float* S, int64_t n, const float* W1, const float* b1, const float* W2, const float* b2,
               float p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits, float* out, int64_t ld_out,
               float* inv_norm, uint8_t* flags, cudaStream_t stream) {
    using C = Cfg<DIN, DOUT>;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(biagg_fwd_kernel<DIN, DOUT>, (int)C::fwd_smem, configured); rc != KGAT_OK) return rc;
    const int grid = grid_for(n, C::TM, C::fwd_smem);
    biagg_fwd_kernel<DIN, DOUT><<<grid, C::NT, C::fwd_smem, stream>>>(E, S, n, W1, b1, W2, b2, p, seed, offset, seed_dev, keep_bits,
                                                                     out, ld_out, inv_norm, flags);
    return check_launch();
}

template <int DIN, int DOUT>
int launch_bwd(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm, const uint8_t* flags,
               const float* E, const float* S, int64_t n, const float* W1, const float* W2, float p, float* g_S, float* g_E,
               float* partials, int n_ctas, cudaStream_t stream) {
    using C = Cfg<DIN, DOUT>;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(biagg_bwd_kernel<DIN, DOUT>, (int)C::bwd_smem, configured); rc != KGAT_OK) return rc;
    biagg_bwd_kernel<DIN, DOUT><<<n_ctas, C::NT, C::bwd_smem, stream>>>(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, n, W1, W2,
                                                                       p, g_S, g_E, partials);
    return check_launch();
}

template <int DIN, int DOUT>
int bwd_ctas(int64_t n) {
    using C = Cfg<DIN, DOUT>;
    return grid_for(n, C::TM, C::bwd_smem);
}

}  // namespace
}  // namespace kgat

#ifndef KGAT_BIAGG_DEFAULT_IMPL
#define KGAT_BIAGG_DEFAULT_IMPL 2
#endif

namespace kgat {
// tensor-core (3xTF32 mma.sync) implementation, biagg_mma.cu
int biagg_mma_forward(const float* E, const float* S, int64_t n, int d_in, int d_out, const float* W1, const float* b1, const float* W2,
                      const float* b2, float p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits,
                      float* out, int64_t ld_out, float* inv_norm, uint8_t* flags, float* const* peer_out, int n_peers,
                      const int32_t* row_ids, const int32_t* n_dev, cudaStream_t stream);
int biagg_mma_backward_ctas(int64_t n, int d_in, int d_out);
int biagg_mma_backward(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm, const uint8_t* flags,
                       const float* E, const float* S, int64_t n, int d_in, int d_out, const float* W1, const float* W2, float p, float* g_S,
                       float* g_E, float* partials, int n_ctas, float* const* peer_gS, int n_peers, const int32_t* row_ids,
                       const int32_t* n_dev, cudaStream_t stream);
// peer.cu: copy n_floats to the same offset behind every peer pointer
int peer_push_launch(const float* src, float* const* peer_dst, int n_peers, int64_t n_floats, cudaStream_t stream, int max_ctas = 0);

// tcgen05 forward (TMEM accumulators), biagg_tc5.cu
bool biagg_tc5_supported(int d_in, int d_out);
int biagg_tc5_forward(const float* E, const float* S, int64_t n, int d_in, int d_out, const float* W1, const float* b1, const float* W2,
                      const float* b2, float p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits,
                      float* out, int64_t ld_out, float* inv_norm, uint8_t* flags, float* const* peer_out, int n_peers,
                      const int32_t* row_ids, const int32_t* n_dev, cudaStream_t stream);

// KGAT_BIAGG_IMPL selects the implementation (A/B comparison): "ffma" = the CUDA-core kernels of this file,
// "mma" = warp-level mma.sync (biagg_mma.cu), "tc5" = tcgen05 forward + mma.sync backward.
static int biagg_impl() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("KGAT_BIAGG_IMPL");
        v = (e == nullptr) ? KGAT_BIAGG_DEFAULT_IMPL : (e[0] == 'f' ? 0 : (e[0] == 't' ? 2 : 1));
    }
    return v;
}
static bool use_mma() { return biagg_impl() >= 1; }
}  // namespace kgat

using namespace kgat;

#define KGAT_DISPATCH_DIMS(DIN_, DOUT_, CALL)                          \
    do {                                                               \
        const int key__ = (DIN_) * 1000 + (DOUT_);                     \
        switch (key__) {                                               \
            case 16016: { constexpr int DI = 16, DO = 16; CALL; }      \
            case 32016: { constexpr int DI = 32, DO = 16; CALL; }      \
            case 32032: { constexpr int DI = 32, DO = 32; CALL; }      \
            case 64016: { constexpr int DI = 64, DO = 16; CALL; }      \
            case 64032: { constexpr int DI = 64, DO = 32; CALL; }      \
            case 64064: { constexpr int DI = 64, DO = 64; CALL; }      \
            case 128064: { constexpr int DI = 128, DO = 64; CALL; }    \
            case 128128: { constexpr int DI = 128, DO = 128; CALL; }   \
            default: return KGAT_ERR_UNSUPPORTED;                      \
        }                                                              \
    } while (0)

extern "C" {

// row_ids / n_dev: optional needed-row list (frontier.cu).  The kernels then run over the *n_dev listed rows (n = the
// list's capacity, used for the grid); every per-row array stays indexed by node id.
static int biagg_forward_impl(const float* E, const float* S, int64_t n, int32_t d_in, int32_t d_out, const float* W1, const float* b1,
                              const float* W2, const float* b2, float dropout_p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                              const uint32_t* keep_bits, float* out, int64_t ld_out, float* inv_norm, uint8_t* flags,
                              float* const* peer_out, int32_t n_peers, const int32_t* row_ids, const int32_t* n_dev, void* stream) {
    if (n < 0 || dropout_p < 0.f || dropout_p >= 1.f || (ld_out & 3) || n_peers < 0 || n_peers > KGAT_MAX_PEERS || (n_peers && !peer_out))
        return KGAT_ERR_INVALID_ARGUMENT;
    if ((row_ids == nullptr) != (n_dev == nullptr)) return KGAT_ERR_INVALID_ARGUMENT;
    if (n == 0) return KGAT_OK;
    if (biagg_impl() == 2 && biagg_tc5_supported(d_in, d_out))
        return biagg_tc5_forward(E, S, n, d_in, d_out, W1, b1, W2, b2, dropout_p, seed, offset, seed_dev, keep_bits, out, ld_out, inv_norm,
                                 flags, peer_out, n_peers, row_ids, n_dev, (cudaStream_t)stream);
    if (use_mma() || row_ids != nullptr)
        return biagg_mma_forward(E, S, n, d_in, d_out, W1, b1, W2, b2, dropout_p, seed, offset, seed_dev, keep_bits, out, ld_out, inv_norm,
                                 flags, peer_out, n_peers, row_ids, n_dev, (cudaStream_t)stream);
    if (n_peers > 0 && ld_out != d_out) return KGAT_ERR_UNSUPPORTED;
    const int rc = [&]() -> int {
        KGAT_DISPATCH_DIMS(d_in, d_out, return (launch_fwd<DI, DO>(E, S, n, W1, b1, W2, b2, dropout_p, seed, offset, seed_dev, keep_bits, out,
                                                                   ld_out, inv_norm, flags, (cudaStream_t)stream)));
    }();
    if (rc != KGAT_OK || n_peers == 0) return rc;
    return peer_push_launch(out, peer_out, n_peers, n * d_out, (cudaStream_t)stream);  // CUDA-core path: unfused push
}

int kgat_biagg_forward(const float* E, const float* S, int64_t n, int32_t d_in, int32_t d_out, const float* W1, const float* b1,
                       const float* W2, const float* b2, float dropout_p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                       const uint32_t* keep_bits, float* out, int64_t ld_out, float* inv_norm, uint8_t* flags, float* const* peer_out,
                       int32_t n_peers, void* stream) {
    return biagg_forward_impl(E, S, n, d_in, d_out, W1, b1, W2, b2, dropout_p, seed, offset, seed_dev, keep_bits, out, ld_out, inv_norm,
                              flags, peer_out, n_peers, nullptr, nullptr, stream);
}

int kgat_biagg_forward_rows(const float* E, const float* S, const int32_t* row_ids, const int32_t* n_rows_dev, int64_t max_rows, int32_t d_in,
                            int32_t d_out, const float* W1, const float* b1, const float* W2, const float* b2, float dropout_p,
                            uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits, float* out, int64_t ld_out,
                            float* inv_norm, uint8_t* flags, void* stream) {
    if (!row_ids || !n_rows_dev) return KGAT_ERR_INVALID_ARGUMENT;
    return biagg_forward_impl(E, S, max_rows, d_in, d_out, W1, b1, W2, b2, dropout_p, seed, offset, seed_dev, keep_bits, out, ld_out,
                              inv_norm, flags, nullptr, 0, row_ids, n_rows_dev, stream);
}

int kgat_biagg_backward_rows_ctas(int64_t max_rows, int32_t d_in, int32_t d_out) {
    if (max_rows <= 0) return 1;
    return biagg_mma_backward_ctas(max_rows, d_in, d_out);  // the row-list backward always runs the tensor-core kernel
}

int kgat_biagg_backward_ctas(int64_t n, int32_t d_in, int32_t d_out) {
    if (n <= 0) return 1;
    if (use_mma()) return biagg_mma_backward_ctas(n, d_in, d_out);
    KGAT_DISPATCH_DIMS(d_in, d_out, return (bwd_ctas<DI, DO>(n)));
}

static int biagg_backward_impl(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm,
                               const uint8_t* flags, const float* E, const float* S, int64_t n, int32_t d_in, int32_t d_out, const float* W1,
                               const float* W2, float dropout_p, float* g_S, float* g_E, float* partials, int32_t n_ctas,
                               float* const* peer_gS, int32_t n_peers, const int32_t* row_ids, const int32_t* n_dev, void* stream) {
    if (n <= 0 || n_ctas <= 0 || (ld_gout & 3) || (ld_out & 3) || n_peers < 0 || n_peers > KGAT_MAX_PEERS || (n_peers && !peer_gS))
        return KGAT_ERR_INVALID_ARGUMENT;
    if ((row_ids == nullptr) != (n_dev == nullptr)) return KGAT_ERR_INVALID_ARGUMENT;
    if (use_mma() || row_ids != nullptr)
        return biagg_mma_backward(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, n, d_in, d_out, W1, W2, dropout_p, g_S, g_E, partials,
                                  n_ctas, peer_gS, n_peers, row_ids, n_dev, (cudaStream_t)stream);
    const int rc = [&]() -> int {
        KGAT_DISPATCH_DIMS(d_in, d_out, return (launch_bwd<DI, DO>(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, n, W1, W2, dropout_p,
                                                                   g_S, g_E, partials, n_ctas, (cudaStream_t)stream)));
    }();
    if (rc != KGAT_OK || n_peers == 0) return rc;
    return peer_push_launch(g_S, peer_gS, n_peers, n * d_in, (cudaStream_t)stream);
}

int kgat_biagg_backward(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm,
                        const uint8_t* flags, const float* E, const float* S, int64_t n, int32_t d_in, int32_t d_out, const float* W1,
                        const float* W2, float dropout_p, float* g_S, float* g_E, float* partials, int32_t n_ctas, float* const* peer_gS,
                        int32_t n_peers, void* stream) {
    return biagg_backward_impl(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, n, d_in, d_out, W1, W2, dropout_p, g_S, g_E, partials,
                               n_ctas, peer_gS, n_peers, nullptr, nullptr, stream);
}

int kgat_biagg_backward_rows(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm,
                             const uint8_t* flags, const float* E, const float* S, const int32_t* row_ids, const int32_t* n_rows_dev,
                             int64_t max_rows, int32_t d_in, int32_t d_out, const float* W1, const float* W2, float dropout_p, float* g_S,
                             float* g_E, float* partials, int32_t n_ctas, void* stream) {
    if (!row_ids || !n_rows_dev) return KGAT_ERR_INVALID_ARGUMENT;
    return biagg_backward_impl(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, max_rows, d_in, d_out, W1, W2, dropout_p, g_S, g_E,
                               partials, n_ctas, nullptr, 0, row_ids, n_rows_dev, stream);
}

int kgat_biagg_reduce_param_grads(const float* partials, int32_t n_ctas, int32_t d_in, int32_t d_out, float* gW1, float* gb1,
                                  float* gW2, float* gb2, int32_t accumulate, void* stream) {
    if (n_ctas <= 0 || d_in <= 0 || d_out <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    const int total = 2 * d_in * d_out + 2 * d_out;
    reduce_partials_kernel<<<(total + 31) / 32, 32 * kReduceParts, 0, (cudaStream_t)stream>>>(partials, n_ctas, d_in, d_out, gW1, gb1, gW2, gb2,
                                                                               accumulate);
    return check_launch();
}

}  // extern "C"
