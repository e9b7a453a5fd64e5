// K2/K3 on the tensor cores: the bi-interaction aggregator's GEMMs as warp-level TF32 MMAs with
// 3xTF32 error compensation (a = hi + lo, a*b ~= lo*hi + hi*lo + hi*hi, fp32 accumulate), which keeps
// the result at fp32-level accuracy (~1e-6 normwise) -- inside the 1e-5 parity budget that plain TF32
// (1e-3) would break.  Same interface, same saved tensors and the same staging / fusion as the FFMA
// kernels in biagg.cu (which remain as the reference implementation, KGAT_BIAGG_IMPL=ffma).
//
// The forward of the shapes with d_in, d_out <= 64 runs on tcgen05 by default (biagg_tc5.cu, TMEM accumulators);
// these warp-level kernels serve the backward, the wider shapes and KGAT_BIAGG_IMPL=mma.  Either way the time
// goes into operand preparation and the epilogue on the CUDA cores, not into the tensor pipe (2.6 GFLOP x 3 per
// layer-forward against 120 MB of traffic); see DESIGN.md section 4.
#include "common.cuh"

namespace kgat {
namespace mma {

__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
// Exact two-term split x = hi + lo with hi representable in TF32.  cvt.rna.tf32 is emulated by ~6 integer
// instructions on sm_100a (ncu: it doubled the instruction count of the MMA loop), so the per-use split
// truncates instead: hi = x with the low 13 mantissa bits cleared (one LOP3), lo = x - hi (exact, one FADD).
// The tensor core ignores the low 13 bits of lo, an error <= 2^-20 |x| per operand (1e-6), which averages
// down across the K-sum and stays inside the 1e-5 budget (tested).  The round-to-nearest variant is used
// where a split is computed once and reused (the weights staged in shared memory).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(x) & 0xffffe000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void split_tf32_rn(float x, uint32_t& hi, uint32_t& lo) {
    hi = to_tf32(x);
    lo = to_tf32(x - __uint_as_float(hi));
}
// D += A (16x8, row) * B (8x8, col), TF32 inputs, fp32 accumulate
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 3xTF32: small cross terms first, then the leading term
__device__ __forceinline__ void mma_3x(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0, uint32_t bh1,
                                       uint32_t bl0, uint32_t bl1) {
    mma_tf32(d, al, bh0, bh1);
    mma_tf32(d, ah, bl0, bl1);
    mma_tf32(d, ah, bh0, bh1);
}

template <int DIN, int DOUT>
struct FwdCfg {
    static constexpr bool kBig = (DIN > 64) || (DOUT > 64);
    static constexpr bool kPreSplit = !kBig;       // weights stored as (hi, lo) TF32 pairs in shared memory
    static constexpr int NT = 256;                 // 8 warps
    static constexpr int TM = 64;                  // rows per CTA tile
    static constexpr int WARPS = NT / 32;
    static constexpr int MT = TM / 16;             // m-tiles per CTA tile
    static constexpr int NTL = DOUT / 8;           // n-tiles
    static constexpr int WPM = WARPS / MT;         // warps sharing one m-tile (2): each takes half of the n-tiles
    static constexpr int NTW = NTL / WPM;          // n-tiles per warp
    static constexpr int SE = DIN + 4;             // smem strides == 4 mod 32: conflict-free fragment reads
    static constexpr int SW = DIN + 4;             // (also == 4 mod 16 for the 8-byte (hi, lo) pairs)
    static constexpr int WELEM = kPreSplit ? 2 : 1;
    static_assert(WARPS % MT == 0 && NTL % WPM == 0 && NTW >= 1, "bad warp mapping");
    static constexpr size_t smem = sizeof(float) * (2 * DOUT * SW * WELEM + 2 * TM * SE + TM * WPM);
};

template <int DIN, int DOUT>
__global__ void __launch_bounds__(256) biagg_fwd_mma_kernel(
    const float* __restrict__ E, const float* __restrict__ S, int64_t n, const float* __restrict__ W1,
    const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2, float dropout_p,
    uint64_t seed, uint64_t offset, const uint64_t* __restrict__ seed_dev, const uint32_t* __restrict__ keep_bits,
    float* __restrict__ out, int64_t ld_out, float* __restrict__ inv_norm, uint8_t* __restrict__ flags,
    float* const* __restrict__ peer_out, int n_peers, const int32_t* __restrict__ row_ids, const int32_t* __restrict__ n_dev) {
    using C = FwdCfg<DIN, DOUT>;
    if (n_dev != nullptr) n = n_dev[0];  // needed-row pruning: run over the listed rows, arrays stay node-indexed
    static_assert(DOUT <= DIN, "the output tile is staged in the E+S tile for the peer stores");
    extern __shared__ __align__(16) float smem[];
    if (seed_dev != nullptr) seed += seed_dev[0] * 0x9E3779B97F4A7C15ull;
    float* W1s = smem;                      // [DOUT][SW] (x2 when pre-split: (hi, lo) pairs)
    float* W2s = W1s + DOUT * C::SW * C::WELEM;
    float* Us = W2s + DOUT * C::SW * C::WELEM;  // [TM][SE]  E + S
    float* Vs = Us + C::TM * C::SE;         // [TM][SE]  E * S
    float* Red = Vs + C::TM * C::SE;        // [TM][WPM] partial row sums
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;

    if (C::kPreSplit) {
        for (int i = tid; i < DOUT * DIN; i += C::NT) {
            const int c = i / DIN, k = i % DIN;
            uint32_t hi, lo;
            split_tf32_rn(W1[i], hi, lo);
            reinterpret_cast<uint2*>(W1s)[c * C::SW + k] = make_uint2(hi, lo);
            split_tf32_rn(W2[i], hi, lo);
            reinterpret_cast<uint2*>(W2s)[c * C::SW + k] = make_uint2(hi, lo);
        }
    } else {
        for (int i = tid; i < DOUT * (DIN / 4); i += C::NT) {
            const int c = i / (DIN / 4), q = i % (DIN / 4);
            *reinterpret_cast<float4*>(W1s + c * C::SW + q * 4) = __ldg(reinterpret_cast<const float4*>(W1 + c * DIN) + q);
            *reinterpret_cast<float4*>(W2s + c * C::SW + q * 4) = __ldg(reinterpret_cast<const float4*>(W2 + c * DIN) + q);
        }
    }
    const int mt = warp % C::MT;            // m-tile of this warp
    const int nw = warp / C::MT;            // which slice of the n-tiles
    const int nt0 = nw * C::NTW;
    const float keep_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    const uint32_t keep_thr = (uint32_t)((1.f - dropout_p) * 65536.f);
    constexpr int words_per_row = (DOUT + 31) / 32;
    const int64_t n_tiles = (n + C::TM - 1) / C::TM;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * C::TM;
        __syncthreads();
        for (int i = tid; i < C::TM * (DIN / 4); i += C::NT) {
            const int r = i / (DIN / 4), q = i % (DIN / 4);
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f), s = e;
            if (row0 + r < n) {
                const int64_t node = row_ids != nullptr ? (int64_t)__ldg(row_ids + row0 + r) : row0 + r;
                e = ld_stream4(E + node * DIN + q * 4);
                s = ld_stream4(S + node * DIN + q * 4);
            }
            *reinterpret_cast<float4*>(Us + r * C::SE + q * 4) = make_float4(e.x + s.x, e.y + s.y, e.z + s.z, e.w + s.w);
            *reinterpret_cast<float4*>(Vs + r * C::SE + q * 4) = make_float4(e.x * s.x, e.y * s.y, e.z * s.z, e.w * s.w);
        }
        __syncthreads();

        float z1[C::NTW][4], z2[C::NTW][4];
#pragma unroll
        for (int j = 0; j < C::NTW; ++j) {
            const int c = (nt0 + j) * 8 + 2 * t;
            z1[j][0] = z1[j][2] = b1[c];
            z1[j][1] = z1[j][3] = b1[c + 1];
            z2[j][0] = z2[j][2] = b2[c];
            z2[j][1] = z2[j][3] = b2[c + 1];
        }
        const float* ua = Us + (mt * 16 + g) * C::SE + t;
        const float* va = Vs + (mt * 16 + g) * C::SE + t;
        // The three TF32 terms of one accumulator are dependent MMAs: issue each term for ALL n-tiles of the
        // warp before the next term so dependent instructions are NTW MMAs apart (hides the HMMA latency).
        for (int ks = 0; ks < DIN / 8; ++ks) {
#pragma unroll
            for (int mat = 0; mat < 2; ++mat) {
                const float* ap = mat == 0 ? ua : va;
                const float* Wm = mat == 0 ? W1s : W2s;
                uint32_t ah[4], al[4], bh0[C::NTW], bh1[C::NTW], bl0[C::NTW], bl1[C::NTW];
                split_tf32(ap[ks * 8], ah[0], al[0]);
                split_tf32(ap[ks * 8 + 8 * C::SE], ah[1], al[1]);
                split_tf32(ap[ks * 8 + 4], ah[2], al[2]);
                split_tf32(ap[ks * 8 + 8 * C::SE + 4], ah[3], al[3]);
#pragma unroll
                for (int j = 0; j < C::NTW; ++j) {
                    const int wrow = ((nt0 + j) * 8 + g) * C::SW + ks * 8 + t;
                    if (C::kPreSplit) {
                        const uint2 p0 = reinterpret_cast<const uint2*>(Wm)[wrow];
                        const uint2 p1 = reinterpret_cast<const uint2*>(Wm)[wrow + 4];
                        bh0[j] = p0.x; bl0[j] = p0.y; bh1[j] = p1.x; bl1[j] = p1.y;
                    } else {
                        split_tf32(Wm[wrow], bh0[j], bl0[j]);
                        split_tf32(Wm[wrow + 4], bh1[j], bl1[j]);
                    }
                }
                if (mat == 0) {
#pragma unroll
                    for (int j = 0; j < C::NTW; ++j) mma_tf32(z1[j], al, bh0[j], bh1[j]);
#pragma unroll
                    for (int j = 0; j < C::NTW; ++j) mma_tf32(z1[j], ah, bl0[j], bl1[j]);
#pragma unroll
                    for (int j = 0; j < C::NTW; ++j) mma_tf32(z1[j], ah, bh0[j], bh1[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < C::NTW; ++j) mma_tf32(z2[j], al, bh0[j], bh1[j]);
#pragma unroll
                    for (int j = 0; j < C::NTW; ++j) mma_tf32(z2[j], ah, bl0[j], bl1[j]);
#pragma unroll
                    for (int j = 0; j < C::NTW; ++j) mma_tf32(z2[j], ah, bh0[j], bh1[j]);
                }
            }
        }

        // epilogue: thread owns rows (mt*16 + g) and (+8), columns (nt0+j)*8 + 2t, +1
        float x[2][C::NTW][2];
        uint8_t f[2][C::NTW][2];
        float ss[2] = {0.f, 0.f};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int64_t idx = row0 + mt * 16 + g + 8 * h;
            const bool valid = idx < n;
            const int64_t row = (valid && row_ids != nullptr) ? (int64_t)__ldg(row_ids + idx) : idx;
            uint32_t rnd[(C::NTW * 2 + 7) / 8 * 4];
            if (dropout_p > 0.f && keep_bits == nullptr && valid) {
#pragma unroll
                for (int q = 0; q < (C::NTW * 2 + 7) / 8; ++q) {
                    const uint4 r4 = philox4x32(seed, offset + ((uint64_t)row * 4 + t) * 8 + nw * 2 + q);
                    rnd[q * 4 + 0] = r4.x; rnd[q * 4 + 1] = r4.y; rnd[q * 4 + 2] = r4.z; rnd[q * 4 + 3] = r4.w;
                }
            }
#pragma unroll
            for (int j = 0; j < C::NTW; ++j) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int c = (nt0 + j) * 8 + 2 * t + e;
                    bool kp = true;
                    if (dropout_p > 0.f && valid) {
                        if (keep_bits != nullptr) {
                            kp = (keep_bits[row * words_per_row + (c >> 5)] >> (c & 31)) & 1u;
                        } else {
                            const int idx = j * 2 + e;  // 16-bit lane of the random words
                            kp = ((rnd[idx >> 1] >> ((idx & 1) * 16)) & 0xffffu) < keep_thr;
                        }
                    }
                    const float a1 = z1[j][2 * h + e], a2 = z2[j][2 * h + e];
                    f[h][j][e] = (a1 > 0.f ? 1 : 0) | (a2 > 0.f ? 2 : 0) | (kp ? 4 : 0);
                    const float v = lrelu(a1) + lrelu(a2);
                    x[h][j][e] = kp ? v * keep_scale : 0.f;
                    ss[h] = fmaf(x[h][j][e], x[h][j][e], ss[h]);
                }
            }
            ss[h] += __shfl_xor_sync(kFull, ss[h], 1);
            ss[h] += __shfl_xor_sync(kFull, ss[h], 2);
        }
        {  // rows are split over WPM warps: combine the partial sums through smem
            if (t == 0) {
                Red[(mt * 16 + g) * C::WPM + nw] = ss[0];
                Red[(mt * 16 + g + 8) * C::WPM + nw] = ss[1];
            }
            __syncthreads();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float tot = 0.f;
#pragma unroll
                for (int q = 0; q < C::WPM; ++q) tot += Red[(mt * 16 + g + 8 * h) * C::WPM + q];
                ss[h] = tot;
            }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int64_t idx = row0 + mt * 16 + g + 8 * h;
            if (idx >= n) continue;
            const int64_t row = row_ids != nullptr ? (int64_t)__ldg(row_ids + idx) : idx;
            const float nrm = sqrtf(ss[h]);
            const float denom = fmaxf(nrm, KGAT_NORM_EPS);
            const float rinv = 1.f / denom;  // one IEEE division per row; x * rinv is within 1 ulp of x / denom
#pragma unroll
            for (int j = 0; j < C::NTW; ++j) {
                const int c = (nt0 + j) * 8 + 2 * t;
                const float2 o = make_float2(x[h][j][0] * rinv, x[h][j][1] * rinv);
                *reinterpret_cast<float2*>(out + row * ld_out + c) = o;
                // every warp is past its MMA loop (barrier above): the E+S tile is free to stage the output rows
                if (n_peers > 0) *reinterpret_cast<float2*>(Us + (mt * 16 + g + 8 * h) * C::SE + c) = o;
                if (flags != nullptr) *reinterpret_cast<uchar2*>(flags + row * DOUT + c) = make_uchar2(f[h][j][0], f[h][j][1]);
            }
            if (inv_norm != nullptr && t == 0 && nw == 0) inv_norm[row] = nrm < KGAT_NORM_EPS ? -rinv : rinv;
        }
        if (n_peers > 0) {
            // row-sharded propagation: the finished rows also go into every peer's copy of the table (NVLink peer
            // stores, 512 B per warp instruction), overlapping the next tile's loads and MMAs
            __syncthreads();
            for (int i = tid; i < C::TM * (DOUT / 4); i += C::NT) {
                const int r = i / (DOUT / 4), q4 = i % (DOUT / 4);
                if (row0 + r < n) {
                    const int64_t node = row_ids != nullptr ? (int64_t)__ldg(row_ids + row0 + r) : row0 + r;
                    const float4 v = *reinterpret_cast<const float4*>(Us + r * C::SE + q4 * 4);
                    for (int q = 0; q < n_peers; ++q) *reinterpret_cast<float4*>(peer_out[q] + node * ld_out + q4 * 4) = v;
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
template <int DIN, int DOUT>
struct BwdCfg {
    static constexpr bool kBig = (DIN > 64) || (DOUT > 64);
    static constexpr int NT = kBig ? 512 : 256;
    static constexpr int WARPS = NT / 32;
    static constexpr int TM = kBig ? 32 : 64;
    static constexpr int SE = DIN + 4;    // E/S tiles: == 4 mod 32 (B operand of the weight-gradient MMA, permuted rows)
    static constexpr int SG = DOUT + 4;   // dL/dz tiles: == 4 mod 32
    static constexpr int SW = DIN + 8;    // weights: == 8 mod 32 (B operand of the input-gradient MMA)
    // phase 1 (elementwise) mapping: CG threads per row
    static constexpr int CG = DOUT / 4;
    static constexpr int RGROUPS = NT / CG;
    static constexpr int RM = (TM + RGROUPS - 1) / RGROUPS;
    // phase 2 (input gradients): output TM x DIN = MT2 x NT2 tiles of 16x8, both products
    static constexpr int MT2 = TM / 16;
    static constexpr int NT2 = DIN / 8;
    static constexpr int TILES2 = MT2 * NT2;
    static constexpr int TPW2 = (TILES2 + WARPS - 1) / WARPS;
    // phase 3 (weight gradients): output DOUT x DIN = MT3 x NT3 tiles, two matrices
    static constexpr int MT3 = DOUT / 16;
    static constexpr int NT3 = DIN / 8;
    static constexpr int TILES3 = 2 * MT3 * NT3;
    static constexpr int TPW3 = (TILES3 + WARPS - 1) / WARPS;
    static constexpr size_t smem = sizeof(float) * (2 * DOUT * SW + 2 * TM * SE + 2 * TM * SG);
};

template <int DIN, int DOUT>
__global__ void __launch_bounds__(BwdCfg<DIN, DOUT>::NT) biagg_bwd_mma_kernel(
    const float* __restrict__ g_out, int64_t ld_gout, const float* __restrict__ out, int64_t ld_out,
    const float* __restrict__ inv_norm, const uint8_t* __restrict__ flags, const float* __restrict__ E,
    const float* __restrict__ S, int64_t n, const float* __restrict__ W1, const float* __restrict__ W2, float dropout_p,
    float* __restrict__ g_S, float* __restrict__ g_E, float* __restrict__ partials, float* const* __restrict__ peer_gS, int n_peers,
    const int32_t* __restrict__ row_ids, const int32_t* __restrict__ n_dev) {
    using C = BwdCfg<DIN, DOUT>;
    if (n_dev != nullptr) n = n_dev[0];  // needed-row pruning: run over the listed rows, arrays stay node-indexed
    extern __shared__ __align__(16) float smem[];
    float* W1s = smem;                    // [DOUT][SW]
    float* W2s = W1s + DOUT * C::SW;
    float* Es = W2s + DOUT * C::SW;       // [TM][SE]
    float* Ss = Es + C::TM * C::SE;
    float* G1 = Ss + C::TM * C::SE;       // [TM][SG]
    float* G2 = G1 + C::TM * C::SG;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;

    for (int i = tid; i < DOUT * (DIN / 4); i += C::NT) {
        const int c = i / (DIN / 4), q = i % (DIN / 4);
        *reinterpret_cast<float4*>(W1s + c * C::SW + q * 4) = __ldg(reinterpret_cast<const float4*>(W1 + c * DIN) + q);
        *reinterpret_cast<float4*>(W2s + c * C::SW + q * 4) = __ldg(reinterpret_cast<const float4*>(W2 + c * DIN) + q);
    }
    const float keep_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    const int cg = tid % C::CG, rg = tid / C::CG;

    // persistent accumulators: weight-gradient tiles of this warp, bias-gradient column of this thread
    float aw[C::TPW3][4];
#pragma unroll
    for (int q = 0; q < C::TPW3; ++q) aw[q][0] = aw[q][1] = aw[q][2] = aw[q][3] = 0.f;
    float ab = 0.f;  // threads [0, DOUT): db1[tid]; [DOUT, 2 DOUT): db2[tid - DOUT]

    const int64_t n_tiles = (n + C::TM - 1) / C::TM;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * C::TM;
        __syncthreads();
        for (int i = tid; i < C::TM * (DIN / 4); i += C::NT) {
            const int r = i / (DIN / 4), q = i % (DIN / 4);
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f), s = e;
            if (row0 + r < n) {
                const int64_t node = row_ids != nullptr ? (int64_t)__ldg(row_ids + row0 + r) : row0 + r;
                e = ld_stream4(E + node * DIN + q * 4);
                s = ld_stream4(S + node * DIN + q * 4);
            }
            *reinterpret_cast<float4*>(Es + r * C::SE + q * 4) = e;
            *reinterpret_cast<float4*>(Ss + r * C::SE + q * 4) = s;
        }
        // ---- phase 1: normalise / dropout / LeakyReLU backward -> dL/dz1, dL/dz2 (all threads run it:
        //      the row reduction is a shuffle over the CG threads of a row) ----
#pragma unroll
        for (int i = 0; i < C::RM; ++i) {
            const int r = rg * C::RM + i;
            const bool in_tile = r < C::TM;
            float4 gg = make_float4(0.f, 0.f, 0.f, 0.f), y = gg;
            uchar4 f = make_uchar4(0, 0, 0, 0);
            float inv = 0.f;
            if (in_tile && row0 + r < n) {
                const int64_t row = row_ids != nullptr ? (int64_t)__ldg(row_ids + row0 + r) : row0 + r;
                gg = ld_stream4(g_out + row * ld_gout + cg * 4);
                y = ld_stream4(out + row * ld_out + cg * 4);
                f = *reinterpret_cast<const uchar4*>(flags + row * DOUT + cg * 4);
                inv = inv_norm[row];
            }
            float tt = gg.x * y.x + gg.y * y.y + gg.z * y.z + gg.w * y.w;
#pragma unroll
            for (int o = 1; o < C::CG; o <<= 1) tt += __shfl_xor_sync(kFull, tt, o);
            if (inv < 0.f) {
                tt = 0.f;
                inv = -inv;
            }
            const float gx[4] = {inv * (gg.x - y.x * tt), inv * (gg.y - y.y * tt), inv * (gg.z - y.z * tt), inv * (gg.w - y.w * tt)};
            const uint8_t fl[4] = {f.x, f.y, f.z, f.w};
            float a1[4], a2[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float gd = (fl[j] & 4) ? gx[j] * keep_scale : 0.f;
                a1[j] = (fl[j] & 1) ? gd : gd * KGAT_LEAKY_SLOPE;
                a2[j] = (fl[j] & 2) ? gd : gd * KGAT_LEAKY_SLOPE;
            }
            if (in_tile) {
                *reinterpret_cast<float4*>(G1 + r * C::SG + cg * 4) = make_float4(a1[0], a1[1], a1[2], a1[3]);
                *reinterpret_cast<float4*>(G2 + r * C::SG + cg * 4) = make_float4(a2[0], a2[1], a2[2], a2[3]);
            }
        }
        __syncthreads();

        // ---- phase 2: input gradients  gu = G1 W1, gv = G2 W2  (M = rows, N = DIN, K = DOUT).
        //      A warp's TPW2 output tiles share the m-tile (WARPS % MT2 == 0), so the G fragments are split once
        //      per c-step and each TF32 term is issued for all 2*TPW2 accumulators before the next term. ----
        {
            static_assert(C::WARPS % C::MT2 == 0 && C::TILES2 % C::WARPS == 0, "phase-2 mapping");
            const int mt = warp % C::MT2;
            const int ntb = warp / C::MT2;                 // first n-tile of this warp
            constexpr int NSTEP = C::WARPS / C::MT2;       // n-tile stride between the warp's tiles
            float gu[C::TPW2][4], gv[C::TPW2][4];
#pragma unroll
            for (int q = 0; q < C::TPW2; ++q) gu[q][0] = gu[q][1] = gu[q][2] = gu[q][3] = gv[q][0] = gv[q][1] = gv[q][2] = gv[q][3] = 0.f;
            const float* a1p = G1 + (mt * 16 + g) * C::SG + t;
            const float* a2p = G2 + (mt * 16 + g) * C::SG + t;
            for (int cs = 0; cs < DOUT / 8; ++cs) {
#pragma unroll
                for (int mat = 0; mat < 2; ++mat) {
                    const float* ap = mat == 0 ? a1p : a2p;
                    const float* Wm = mat == 0 ? W1s : W2s;
                    uint32_t ah[4], al[4], bh0[C::TPW2], bh1[C::TPW2], bl0[C::TPW2], bl1[C::TPW2];
                    split_tf32(ap[cs * 8], ah[0], al[0]);
                    split_tf32(ap[cs * 8 + 8 * C::SG], ah[1], al[1]);
                    split_tf32(ap[cs * 8 + 4], ah[2], al[2]);
                    split_tf32(ap[cs * 8 + 8 * C::SG + 4], ah[3], al[3]);
#pragma unroll
                    for (int q = 0; q < C::TPW2; ++q) {
                        const int wrow = (cs * 8 + t) * C::SW + (ntb + q * NSTEP) * 8 + g;  // B[k = c][n = k_in] = W[c][k_in]
                        split_tf32(Wm[wrow], bh0[q], bl0[q]);
                        split_tf32(Wm[wrow + 4 * C::SW], bh1[q], bl1[q]);
                    }
                    if (mat == 0) {
#pragma unroll
                        for (int q = 0; q < C::TPW2; ++q) mma_tf32(gu[q], al, bh0[q], bh1[q]);
#pragma unroll
                        for (int q = 0; q < C::TPW2; ++q) mma_tf32(gu[q], ah, bl0[q], bl1[q]);
#pragma unroll
                        for (int q = 0; q < C::TPW2; ++q) mma_tf32(gu[q], ah, bh0[q], bh1[q]);
                    } else {
#pragma unroll
                        for (int q = 0; q < C::TPW2; ++q) mma_tf32(gv[q], al, bh0[q], bh1[q]);
#pragma unroll
                        for (int q = 0; q < C::TPW2; ++q) mma_tf32(gv[q], ah, bl0[q], bl1[q]);
#pragma unroll
                        for (int q = 0; q < C::TPW2; ++q) mma_tf32(gv[q], ah, bh0[q], bh1[q]);
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < C::TPW2; ++q) {
                const int nt = ntb + q * NSTEP;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int r = mt * 16 + g + 8 * h;
                    if (row0 + r < n) {
                        const int64_t row = row_ids != nullptr ? (int64_t)__ldg(row_ids + row0 + r) : row0 + r;
                        const int k = nt * 8 + 2 * t;
                        const float2 e = *reinterpret_cast<const float2*>(Es + r * C::SE + k);
                        const float2 s2 = *reinterpret_cast<const float2*>(Ss + r * C::SE + k);
                        // u = E + S, v = E * S:  dS = gu + gv * E,  dE = gu + gv * S
                        const float2 gs = make_float2(fmaf(gv[q][2 * h], e.x, gu[q][2 * h]), fmaf(gv[q][2 * h + 1], e.y, gu[q][2 * h + 1]));
                        *reinterpret_cast<float2*>(g_S + row * DIN + k) = gs;
                        for (int pq = 0; pq < n_peers; ++pq) *reinterpret_cast<float2*>(peer_gS[pq] + row * DIN + k) = gs;
                        *reinterpret_cast<float2*>(g_E + row * DIN + k) =
                            make_float2(fmaf(gv[q][2 * h], s2.x, gu[q][2 * h]), fmaf(gv[q][2 * h + 1], s2.y, gu[q][2 * h + 1]));
                    }
                }
            }
        }

        // ---- phase 3: weight gradients  dW1 += G1^T (E+S),  dW2 += G2^T (E*S)  (M = c, N = k_in, K = rows).
        //      The k index j of an 8-row step maps to row 2j (j<4) / 2(j-4)+1 (j>=4): with strides == 4 mod 32
        //      this permutation makes both fragment reads bank-conflict free; A and B use the same map.
        //      Tile list: tl = warp + q*WARPS over [mat][nt][mt]; each TF32 term is issued for all of the
        //      warp's TPW3 accumulators before the next term. ----
        for (int rs = 0; rs < C::TM / 8; ++rs) {
            const int ra = rs * 8 + 2 * t;      // k = t      -> row 2t
            const int rb = rs * 8 + 2 * t + 1;  // k = t + 4  -> row 2t + 1
            uint32_t bh0[C::TPW3], bh1[C::TPW3], bl0[C::TPW3], bl1[C::TPW3];
            // the warp's tiles of one matrix share the m-tile when WARPS % MT3 == 0: split G once per matrix
            constexpr bool kShareA = (C::WARPS % C::MT3 == 0) && (C::TPW3 % 2 == 0) && (C::TILES3 % C::WARPS == 0);
            uint32_t ah[kShareA ? 2 : C::TPW3][4], al[kShareA ? 2 : C::TPW3][4];
#pragma unroll
            for (int q = 0; q < C::TPW3; ++q) {
                const int tl = warp + q * C::WARPS;
                if (tl < C::TILES3) {
                    const int mat = tl / (C::MT3 * C::NT3);
                    const int rem = tl % (C::MT3 * C::NT3);
                    const int mt = rem % C::MT3, nt = rem / C::MT3;
                    const float* Gm = mat == 0 ? G1 : G2;
                    const int ai = kShareA ? (q / (C::TPW3 / 2)) : q;
                    if (!kShareA || (q % (C::TPW3 / 2)) == 0) {
                        split_tf32(Gm[ra * C::SG + mt * 16 + g], ah[ai][0], al[ai][0]);
                        split_tf32(Gm[ra * C::SG + mt * 16 + g + 8], ah[ai][1], al[ai][1]);
                        split_tf32(Gm[rb * C::SG + mt * 16 + g], ah[ai][2], al[ai][2]);
                        split_tf32(Gm[rb * C::SG + mt * 16 + g + 8], ah[ai][3], al[ai][3]);
                    }
                    const float e0 = Es[ra * C::SE + nt * 8 + g], s0 = Ss[ra * C::SE + nt * 8 + g];
                    const float e1 = Es[rb * C::SE + nt * 8 + g], s1 = Ss[rb * C::SE + nt * 8 + g];
                    split_tf32(mat == 0 ? e0 + s0 : e0 * s0, bh0[q], bl0[q]);
                    split_tf32(mat == 0 ? e1 + s1 : e1 * s1, bh1[q], bl1[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < C::TPW3; ++q)
                if (warp + q * C::WARPS < C::TILES3) mma_tf32(aw[q], al[kShareA ? (q / (C::TPW3 / 2)) : q], bh0[q], bh1[q]);
#pragma unroll
            for (int q = 0; q < C::TPW3; ++q)
                if (warp + q * C::WARPS < C::TILES3) mma_tf32(aw[q], ah[kShareA ? (q / (C::TPW3 / 2)) : q], bl0[q], bl1[q]);
#pragma unroll
            for (int q = 0; q < C::TPW3; ++q)
                if (warp + q * C::WARPS < C::TILES3) mma_tf32(aw[q], ah[kShareA ? (q / (C::TPW3 / 2)) : q], bh0[q], bh1[q]);
        }
        if (tid < 2 * DOUT) {
            const float* Gm = tid < DOUT ? G1 : G2;
            const int c = tid < DOUT ? tid : tid - DOUT;
            float sacc = 0.f;
#pragma unroll 8
            for (int r = 0; r < C::TM; ++r) sacc += Gm[r * C::SG + c];
            ab += sacc;
        }
    }

    // per-CTA partials: [dW1 (DOUT x DIN)][dW2][db1 (DOUT)][db2]
    float* p = partials + (int64_t)blockIdx.x * (2 * DIN * DOUT + 2 * DOUT);
#pragma unroll
    for (int q = 0; q < C::TPW3; ++q) {
        const int tl = warp + q * C::WARPS;
        if (tl >= C::TILES3) break;
        const int mat = tl / (C::MT3 * C::NT3);
        const int rem = tl % (C::MT3 * C::NT3);
        const int mt = rem % C::MT3, nt = rem / C::MT3;
        float* dst = p + mat * DIN * DOUT;
        const int c = mt * 16 + g, k = nt * 8 + 2 * t;
        *reinterpret_cast<float2*>(dst + c * DIN + k) = make_float2(aw[q][0], aw[q][1]);
        *reinterpret_cast<float2*>(dst + (c + 8) * DIN + k) = make_float2(aw[q][2], aw[q][3]);
    }
    if (tid < 2 * DOUT) p[2 * DIN * DOUT + tid] = ab;
}

inline int grid_for(int64_t n, int tm, size_t smem_bytes) {
    const int64_t tiles = (n + tm - 1) / tm;
    int per_sm = (int)(220 * 1024 / (smem_bytes + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 3) per_sm = 3;
    const int64_t cap = (int64_t)sm_count() * per_sm;
    return (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
}

template <int DIN, int DOUT>
int launch_fwd(const float* E, const float* S, int64_t n, const float* W1, const float* b1, const float* W2, const float* b2,
               float p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits, float* out, int64_t ld_out,
               float* inv_norm, uint8_t* flags, float* const* peer_out, int n_peers, const int32_t* row_ids, const int32_t* n_dev,
               cudaStream_t stream) {
    using C = FwdCfg<DIN, DOUT>;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(biagg_fwd_mma_kernel<DIN, DOUT>, (int)C::smem, configured); rc != KGAT_OK) return rc;
    biagg_fwd_mma_kernel<DIN, DOUT><<<grid_for(n, C::TM, C::smem), C::NT, C::smem, stream>>>(E, S, n, W1, b1, W2, b2, p, seed, offset, seed_dev,
                                                                                         keep_bits, out, ld_out, inv_norm, flags, peer_out,
                                                                                         n_peers, row_ids, n_dev);
    return check_launch();
}

template <int DIN, int DOUT>
int launch_bwd(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm, const uint8_t* flags,
               const float* E, const float* S, int64_t n, const float* W1, const float* W2, float p, float* g_S, float* g_E,
               float* partials, int n_ctas, float* const* peer_gS, int n_peers, const int32_t* row_ids, const int32_t* n_dev,
               cudaStream_t stream) {
    using C = BwdCfg<DIN, DOUT>;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(biagg_bwd_mma_kernel<DIN, DOUT>, (int)C::smem, configured); rc != KGAT_OK) return rc;
    biagg_bwd_mma_kernel<DIN, DOUT><<<n_ctas, C::NT, C::smem, stream>>>(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, n, W1, W2, p, g_S,
                                                                    g_E, partials, peer_gS, n_peers, row_ids, n_dev);
    return check_launch();
}

}  // namespace mma

#define KGAT_MMA_DISPATCH(DIN_, DOUT_, CALL)                           \
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

int biagg_mma_forward(const float* E, const float* S, int64_t n, int d_in, int d_out, const float* W1, const float* b1, const float* W2,
                      const float* b2, float p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits,
                      float* out, int64_t ld_out, float* inv_norm, uint8_t* flags, float* const* peer_out, int n_peers,
                      const int32_t* row_ids, const int32_t* n_dev, cudaStream_t stream) {
    KGAT_MMA_DISPATCH(d_in, d_out, return (mma::launch_fwd<DI, DO>(E, S, n, W1, b1, W2, b2, p, seed, offset, seed_dev, keep_bits, out, ld_out,
                                                                   inv_norm, flags, peer_out, n_peers, row_ids, n_dev, stream)));
}

int biagg_mma_backward_ctas(int64_t n, int d_in, int d_out) {
    KGAT_MMA_DISPATCH(d_in, d_out, return (mma::grid_for(n, mma::BwdCfg<DI, DO>::TM, mma::BwdCfg<DI, DO>::smem)));
}

int biagg_mma_backward(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm, const uint8_t* flags,
                       const float* E, const float* S, int64_t n, int d_in, int d_out, const float* W1, const float* W2, float p, float* g_S,
                       float* g_E, float* partials, int n_ctas, float* const* peer_gS, int n_peers, const int32_t* row_ids,
                       const int32_t* n_dev, cudaStream_t stream) {
    KGAT_MMA_DISPATCH(d_in, d_out, return (mma::launch_bwd<DI, DO>(g_out, ld_gout, out, ld_out, inv_norm, flags, E, S, n, W1, W2, p, g_S, g_E,
                                                                   partials, n_ctas, peer_gS, n_peers, row_ids, n_dev, stream)));
}

}  // namespace kgat
