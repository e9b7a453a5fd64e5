// K2 on the 5th-generation tensor cores: the bi-interaction aggregator forward (reference aggregator.py:57-65)
// with tcgen05.mma (kind::tf32, 3xTF32 error compensation) and the two accumulators in tensor memory.
//
//   z1 = (E + S) W1^T + b1,  z2 = (E * S) W2^T + b2,  x = dropout(lrelu(z1) + lrelu(z2)),  out = x / max(||x||, eps)
//
// One persistent CTA per SM, 512 threads (256 for DOUT = 16), 128-row tiles:
//   produce   all 8 warps load the E / S rows of the tile, form U = E + S and V = E * S, split them into TF32-exact
//             hi and lo parts and store the four operand tiles in shared memory in the canonical K-major
//             (no-swizzle) UMMA layout: 8-row x 16-byte core matrices, 128 B apart along K, KC * 128 B apart along M;
//   mma       one thread issues, per product, lo*hi + hi*lo + hi*hi as DIN/8 K-steps each (M = 128, N = DOUT, K = 8)
//             into D1 = TMEM columns [0, DOUT) and D2 = [DOUT, 2 DOUT) of one of TWO accumulator sets, then commits to
//             an mbarrier;
//   epilogue  thread (lane quadrant q = warp % 4, column slice h = warp / 4) owns row 32 q + lane and DOUT / NQ columns:
//             tcgen05.ld, bias, LeakyReLU, dropout, row norm (the two halves meet through shared memory), stores.
// Software pipeline (shared memory holds ONE set of operand tiles, 193 KB with the weights, so one CTA per SM and no
// second CTA to hide latencies): the E / S values of tile i+1 are loaded into registers a whole tile ahead; as soon as
// tile i's MMAs have completed, tile i+1's operands are staged and its MMAs issued into the other accumulator set,
// and they run underneath tile i's epilogue.
// The operand tiles are not plain copies of global memory (they are computed and split), so they are produced by the
// CTA itself rather than by TMA; the weights are split and staged once per CTA.
//
// Accuracy: hi parts are exact TF32 values (low 13 mantissa bits cleared), lo = x - hi is exact in fp32 and the
// tensor core keeps its top 11 bits: the dropped term is <= 2^-21 |x| per operand, as in biagg_mma.cu.
#include "common.cuh"

namespace kgat {
namespace tc5 {

template <int DIN, int DOUT>
struct Cfg {
    static constexpr int TM = 128;
    static constexpr int NT = DOUT >= 32 ? 512 : 256;  // 16 warps where the tile has the columns to occupy them
    static constexpr int NQ = NT / 128;                // column slices per row in the epilogue (warp / 4)
    static constexpr int KC = DIN / 4;                 // 16-byte chunks along K
    static constexpr int A_TILE = TM * DIN;            // floats per A operand tile
    static constexpr int W_TILE = DOUT * DIN;          // floats per B operand tile
    static constexpr int SBO = KC * 128;               // bytes between 8-row groups
    static constexpr int LBO = 128;                    // bytes between K chunks (core matrices)
    static constexpr int COLS = 4 * DOUT <= 64 ? 64 : (4 * DOUT <= 128 ? 128 : 256);  // TMEM columns: two accumulator sets
    static constexpr int CH = DOUT / NQ;               // output columns per epilogue thread
    static constexpr size_t smem = sizeof(float) * (4 * A_TILE + 4 * W_TILE + NQ * TM + 2 * DOUT) + 32;
    static_assert(DIN % 8 == 0 && DOUT % 16 == 0 && DOUT >= 16 && DOUT <= 64 && DIN <= 64, "unsupported tile shape");
    static_assert(CH % 8 == 0, "epilogue loads 8 columns at a time");
};

// element (row r, 16-byte chunk q) of an operand tile, in floats
template <int KC>
__device__ __forceinline__ int canon(int r, int q) {
    return (r >> 3) * (KC * 32) + q * 32 + (r & 7) * 4;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor: K-major, no swizzle, Blackwell descriptor version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(lbo_bytes >> 4) << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// instruction descriptor: D = F32, A = B = TF32, both K-major, N >> 3, M >> 4
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (long long spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (spin > (1ll << 28)) __trap();  // a lost commit must not hang the GPU
    }
}

template <int DIN, int DOUT>
__global__ void __launch_bounds__(Cfg<DIN, DOUT>::NT, 1) biagg_fwd_tc5_kernel(
    const float* __restrict__ E, const float* __restrict__ S, int64_t n, const float* __restrict__ W1, const float* __restrict__ b1,
    const float* __restrict__ W2, const float* __restrict__ b2, float dropout_p, uint64_t seed, uint64_t offset,
    const uint64_t* __restrict__ seed_dev, const uint32_t* __restrict__ keep_bits, float* __restrict__ out, int64_t ld_out,
    float* __restrict__ inv_norm, uint8_t* __restrict__ flags, float* const* __restrict__ peer_out, int n_peers,
    const int32_t* __restrict__ row_ids, const int32_t* __restrict__ n_dev) {
    // row_ids / n_dev (needed-row pruning, frontier.cu): the kernel runs over the *n_dev listed rows; every per-row
    // array (E, S, out, inv_norm, flags, keep_bits, the dropout stream) is still indexed by the node id row_ids[i]
    using C = Cfg<DIN, DOUT>;
    if (n_dev != nullptr) n = n_dev[0];
    extern __shared__ __align__(128) float smem[];
    float* At = smem;                          // [4][A_TILE]: U hi, U lo, V hi, V lo
    float* Wt = At + 4 * C::A_TILE;            // [4][W_TILE]: W1 hi, W1 lo, W2 hi, W2 lo
    float* Red = Wt + 4 * C::W_TILE;           // [TM][NQ]
    float* Bs = Red + C::NQ * C::TM;           // [2][DOUT] biases
    uint64_t* mbar = reinterpret_cast<uint64_t*>(Bs + 2 * DOUT);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 1);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (seed_dev != nullptr) seed += seed_dev[0] * 0x9E3779B97F4A7C15ull;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(C::COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 2 * DOUT; i += C::NT) Bs[i] = i < DOUT ? b1[i] : b2[i - DOUT];
    // weights: split once, canonical layout (row = output column c, K = input feature)
    for (int i = tid; i < DOUT * C::KC; i += C::NT) {
        const int c_lo = i & 7, q = (i >> 3) % C::KC, c_hi = i / (8 * C::KC);
        const int c = c_hi * 8 + c_lo;
        const int o = canon<C::KC>(c, q);
#pragma unroll
        for (int mat = 0; mat < 2; ++mat) {
            const float4 w = __ldg(reinterpret_cast<const float4*>((mat == 0 ? W1 : W2) + c * DIN) + q);
            float4 hi, lo;
            hi.x = __uint_as_float(__float_as_uint(w.x) & 0xffffe000u); lo.x = w.x - hi.x;
            hi.y = __uint_as_float(__float_as_uint(w.y) & 0xffffe000u); lo.y = w.y - hi.y;
            hi.z = __uint_as_float(__float_as_uint(w.z) & 0xffffe000u); lo.z = w.z - hi.z;
            hi.w = __uint_as_float(__float_as_uint(w.w) & 0xffffe000u); lo.w = w.w - hi.w;
            *reinterpret_cast<float4*>(Wt + (2 * mat) * C::W_TILE + o) = hi;
            *reinterpret_cast<float4*>(Wt + (2 * mat + 1) * C::W_TILE + o) = lo;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t bar = smem_u32(mbar);
    const uint32_t a_base = smem_u32(At), w_base = smem_u32(Wt);
    constexpr uint32_t idesc = make_idesc(C::TM, DOUT);

    const int lq = warp & 3, half = warp >> 2;  // lane quadrant of the tile, column slice of the row
    const int r_tile = lq * 32 + lane;  // row of the tile this thread finishes
    const float keep_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    const uint32_t keep_thr = (uint32_t)((1.f - dropout_p) * 65536.f);
    constexpr int words_per_row = (DOUT + 31) / 32;
    const int64_t n_tiles = (n + C::TM - 1) / C::TM;
    constexpr int PF = C::TM * C::KC / C::NT;  // (row, chunk) pairs per thread and tile
    static_assert(C::TM * C::KC % C::NT == 0, "tile must divide evenly over the threads");
    float4 pe[PF], ps[PF];                     // the next tile's E / S values, in flight while this tile is finished

    // global -> registers (issued a whole tile ahead so the HBM latency hides behind the MMA and the epilogue)
    auto prefetch = [&](int64_t tile) {
        const int64_t row0 = tile * C::TM;
#pragma unroll
        for (int it = 0; it < PF; ++it) {
            const int i = tid + it * C::NT;
            const int r = (i / (8 * C::KC)) * 8 + (i & 7), q = (i >> 3) % C::KC;
            pe[it] = ps[it] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (tile < n_tiles && row0 + r < n) {
                const int64_t node = row_ids != nullptr ? (int64_t)__ldg(row_ids + row0 + r) : row0 + r;
                pe[it] = ld_stream4(E + node * DIN + q * 4);
                ps[it] = ld_stream4(S + node * DIN + q * 4);
            }
        }
    };
    // registers -> the four operand tiles (U = E + S and V = E * S, each split into TF32-exact hi and lo)
    auto stage = [&]() {
#pragma unroll
        for (int it = 0; it < PF; ++it) {
            const int i = tid + it * C::NT;
            const int r = (i / (8 * C::KC)) * 8 + (i & 7), q = (i >> 3) % C::KC;
            const float4 e = pe[it], s4 = ps[it];
            const float4 u = make_float4(e.x + s4.x, e.y + s4.y, e.z + s4.z, e.w + s4.w);
            const float4 v = make_float4(e.x * s4.x, e.y * s4.y, e.z * s4.z, e.w * s4.w);
            float4 uh, ul, vh, vl;
            uh.x = __uint_as_float(__float_as_uint(u.x) & 0xffffe000u); ul.x = u.x - uh.x;
            uh.y = __uint_as_float(__float_as_uint(u.y) & 0xffffe000u); ul.y = u.y - uh.y;
            uh.z = __uint_as_float(__float_as_uint(u.z) & 0xffffe000u); ul.z = u.z - uh.z;
            uh.w = __uint_as_float(__float_as_uint(u.w) & 0xffffe000u); ul.w = u.w - uh.w;
            vh.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u); vl.x = v.x - vh.x;
            vh.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u); vl.y = v.y - vh.y;
            vh.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u); vl.z = v.z - vh.z;
            vh.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u); vl.w = v.w - vh.w;
            const int o = canon<C::KC>(r, q);
            *reinterpret_cast<float4*>(At + 0 * C::A_TILE + o) = uh;
            *reinterpret_cast<float4*>(At + 1 * C::A_TILE + o) = ul;
            *reinterpret_cast<float4*>(At + 2 * C::A_TILE + o) = vh;
            *reinterpret_cast<float4*>(At + 3 * C::A_TILE + o) = vl;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the tensor core
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
    };
    // one thread: 2 products x 3 terms x DIN/8 K-steps into accumulator set `buf`, then commit to the mbarrier.
    // The eight operand descriptors are loop invariants; a K-step only advances the 14-bit start-address field.
    uint64_t a_desc[4], b_desc[4];
#pragma unroll
    for (int t4 = 0; t4 < 4; ++t4) {
        a_desc[t4] = make_desc(a_base + t4 * C::A_TILE * 4, C::LBO, C::SBO);
        b_desc[t4] = make_desc(w_base + t4 * C::W_TILE * 4, C::LBO, C::SBO);
    }
    auto issue = [&](int buf) {
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int mat = 0; mat < 2; ++mat) {
                const uint32_t d_tmem = tmem_base + buf * 2 * DOUT + mat * DOUT;
                const int a_sel[3] = {2 * mat + 1, 2 * mat, 2 * mat};  // lo*hi, hi*lo, hi*hi: small terms first
                const int b_sel[3] = {2 * mat, 2 * mat + 1, 2 * mat};
#pragma unroll
                for (int term = 0; term < 3; ++term) {
#pragma unroll
                    for (int ks = 0; ks < DIN / 8; ++ks)
                        mma_tf32_ss(d_tmem, a_desc[a_sel[term]] + (uint64_t)(ks * 16), b_desc[b_sel[term]] + (uint64_t)(ks * 16), idesc,
                                    (term | ks) != 0 ? 1u : 0u);
                }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
        }
    };

    uint32_t parity = 0;
    int buf = 0;
    int64_t tile = blockIdx.x;
    if (tile < n_tiles) {
        prefetch(tile);
        stage();
        issue(0);
        prefetch(tile + gridDim.x);
    }
    for (; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
        const int64_t row0 = tile * C::TM;
        mbar_wait(bar, parity);  // this tile's accumulators are complete and the operand tiles are free again
        parity ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (tile + gridDim.x < n_tiles) {  // next tile: operands from the prefetched registers, MMAs run under this epilogue
            stage();
            issue(buf ^ 1);
            prefetch(tile + 2 * (int64_t)gridDim.x);
        }

        // ---- epilogue: this thread's row, columns [half * CH, half * CH + CH)
        const bool valid = row0 + r_tile < n;
        const int64_t row = (valid && row_ids != nullptr) ? (int64_t)__ldg(row_ids + row0 + r_tile) : row0 + r_tile;
        uint32_t z1[C::CH], z2[C::CH];
        const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + buf * 2 * DOUT + half * C::CH;
#pragma unroll
        for (int j = 0; j < C::CH / 8; ++j) {
            tmem_ld8(taddr + j * 8, z1 + j * 8);
            tmem_ld8(taddr + DOUT + j * 8, z2 + j * 8);
        }
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        float x[C::CH];
        uint32_t fl[C::CH / 4];  // 4 flag bytes per word
        float ss = 0.f;
        uint32_t rnd[C::CH / 8 * 4];
        if (dropout_p > 0.f && keep_bits == nullptr && valid) {
#pragma unroll
            for (int q = 0; q < C::CH / 8; ++q) {
                const uint4 r4 = philox4x32(seed, offset + (uint64_t)row * 32 + half * 4 + q);
                rnd[q * 4 + 0] = r4.x; rnd[q * 4 + 1] = r4.y; rnd[q * 4 + 2] = r4.z; rnd[q * 4 + 3] = r4.w;
            }
        }
#pragma unroll
        for (int j = 0; j < C::CH; ++j) {
            const int c = half * C::CH + j;
            bool kp = true;
            if (dropout_p > 0.f && valid) {
                if (keep_bits != nullptr) kp = (keep_bits[row * words_per_row + (c >> 5)] >> (c & 31)) & 1u;
                else kp = ((rnd[j >> 1] >> ((j & 1) * 16)) & 0xffffu) < keep_thr;
            }
            const float a1 = __uint_as_float(z1[j]) + Bs[c], a2 = __uint_as_float(z2[j]) + Bs[DOUT + c];
            const uint32_t f = (a1 > 0.f ? 1u : 0u) | (a2 > 0.f ? 2u : 0u) | (kp ? 4u : 0u);
            if ((j & 3) == 0) fl[j >> 2] = f; else fl[j >> 2] |= f << (8 * (j & 3));
            const float v = lrelu(a1) + lrelu(a2);
            x[j] = kp ? v * keep_scale : 0.f;
            ss = fmaf(x[j], x[j], ss);
        }
        Red[r_tile * C::NQ + half] = ss;
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();  // the two halves of every row meet; every thread is done reading this accumulator set
        if (valid) {
            float tot = 0.f;
#pragma unroll
            for (int q = 0; q < C::NQ; ++q) tot += Red[r_tile * C::NQ + q];
            const float nrm = sqrtf(tot);
            const float denom = fmaxf(nrm, KGAT_NORM_EPS);
            const float rinv = 1.f / denom;
            float* orow = out + row * ld_out + half * C::CH;
#pragma unroll
            for (int j = 0; j < C::CH; j += 4) {
                const float4 o4 = make_float4(x[j] * rinv, x[j + 1] * rinv, x[j + 2] * rinv, x[j + 3] * rinv);
                *reinterpret_cast<float4*>(orow + j) = o4;
                for (int pq = 0; pq < n_peers; ++pq)
                    *reinterpret_cast<float4*>(peer_out[pq] + row * ld_out + half * C::CH + j) = o4;
            }
            if (flags != nullptr) {
                uint32_t* frow = reinterpret_cast<uint32_t*>(flags + row * DOUT + half * C::CH);
#pragma unroll
                for (int j = 0; j < C::CH / 4; ++j) frow[j] = fl[j];
            }
            if (inv_norm != nullptr && half == 0) inv_norm[row] = nrm < KGAT_NORM_EPS ? -rinv : rinv;
        }
        __syncthreads();  // Red is reused by the next tile
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::COLS) : "memory");
}

template <int DIN, int DOUT>
int launch_fwd(const float* E, const float* S, int64_t n, const float* W1, const float* b1, const float* W2, const float* b2, float p,
               uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits, float* out, int64_t ld_out,
               float* inv_norm, uint8_t* flags, float* const* peer_out, int n_peers, const int32_t* row_ids, const int32_t* n_dev,
               cudaStream_t stream) {
    using C = Cfg<DIN, DOUT>;
    static uint64_t configured = 0;
    if (const int rc = raise_smem_limit(biagg_fwd_tc5_kernel<DIN, DOUT>, (int)C::smem, configured); rc != KGAT_OK) return rc;
    const int64_t tiles = (n + C::TM - 1) / C::TM;
    const int grid = (int)(tiles < sm_count() ? tiles : sm_count());
    biagg_fwd_tc5_kernel<DIN, DOUT><<<grid, C::NT, C::smem, stream>>>(E, S, n, W1, b1, W2, b2, p, seed, offset, seed_dev, keep_bits, out,
                                                                   ld_out, inv_norm, flags, peer_out, n_peers, row_ids, n_dev);
    return check_launch();
}

}  // namespace tc5

bool biagg_tc5_supported(int d_in, int d_out) {
    return (d_in == 64 && (d_out == 64 || d_out == 32 || d_out == 16)) || (d_in == 32 && (d_out == 32 || d_out == 16)) ||
           (d_in == 16 && d_out == 16);
}

int biagg_tc5_forward(const float* E, const float* S, int64_t n, int d_in, int d_out, const float* W1, const float* b1, const float* W2,
                      const float* b2, float p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits,
                      float* out, int64_t ld_out, float* inv_norm, uint8_t* flags, float* const* peer_out, int n_peers,
                      const int32_t* row_ids, const int32_t* n_dev, cudaStream_t stream) {
#define KGAT_TC5_CASE(DI, DO)                                                                                                          \
    if (d_in == DI && d_out == DO)                                                                                                     \
        return tc5::launch_fwd<DI, DO>(E, S, n, W1, b1, W2, b2, p, seed, offset, seed_dev, keep_bits, out, ld_out, inv_norm, flags,     \
                                       peer_out, n_peers, row_ids, n_dev, stream);
    KGAT_TC5_CASE(64, 64)
    KGAT_TC5_CASE(64, 32)
    KGAT_TC5_CASE(64, 16)
    KGAT_TC5_CASE(32, 32)
    KGAT_TC5_CASE(32, 16)
    KGAT_TC5_CASE(16, 16)
#undef KGAT_TC5_CASE
    return KGAT_ERR_UNSUPPORTED;
}

}  // namespace kgat
