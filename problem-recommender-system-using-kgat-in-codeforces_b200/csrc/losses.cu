// K4: fused BPR loss over the per-layer embedding tables (reference model.py:189-202, 142-163)
// K5: fused TransR loss without materialising W_r[rel] (reference model.py:204-261)
// Both with hand-written backward kernels.  One warp per sample; the per-sample terms go to a small
// scratch and are reduced in a fixed order by a single-CTA kernel (deterministic loss value).
#include "common.cuh"

namespace kgat {
namespace {

// loss = mean_b(-logsigmoid(margin_b)) + reg * mean_b(l2_b);   scratch = [margin (B)][l2 (B)]
// `pub` (optional): the loss is also published to the host -- ring[s % n_slots] = (s << 32) | bits(loss) with s = ++serial, one
// aligned 8-byte store into mapped pinned memory (what kgat_publish_loss does as a launch of its own)
struct Publish {
    unsigned long long* serial_dev;
    volatile unsigned long long* ring_host;
    int n_slots;
};

// run by one block of 256 threads: loss_reduce_kernel, or the last block of transr_reduce_kernel
__device__ __forceinline__ void loss_reduce(const float* __restrict__ scratch, int batch, float reg, float* __restrict__ loss,
                                            float* __restrict__ loss_sum, Publish pub) {
    __shared__ float sh_a[8], sh_b[8];
    float a = 0.f, b = 0.f;
    for (int i = threadIdx.x; i < batch; i += 256) {
        a += -log_sigmoid(scratch[i]);
        b += scratch[batch + i];
    }
    a = warp_sum(a);
    b = warp_sum(b);
    if ((threadIdx.x & 31) == 0) {
        sh_a[threadIdx.x >> 5] = a;
        sh_b[threadIdx.x >> 5] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float ta = 0.f, tb = 0.f;
        for (int w = 0; w < 8; ++w) {
            ta += sh_a[w];
            tb += sh_b[w];
        }
        const float l = ta / (float)batch + reg * (tb / (float)batch);
        loss[0] = l;
        if (loss_sum != nullptr) loss_sum[0] += l;
        if (pub.serial_dev != nullptr) {
            const unsigned long long sn = pub.serial_dev[0] + 1ull;
            pub.serial_dev[0] = sn;
            pub.ring_host[sn % (unsigned long long)pub.n_slots] = (sn << 32) | (unsigned long long)__float_as_uint(l);
            __threadfence_system();
        }
    }
}

__global__ void __launch_bounds__(256) loss_reduce_kernel(const float* __restrict__ scratch, int batch, float reg,
                                                          float* __restrict__ loss, float* __restrict__ loss_sum = nullptr,
                                                          Publish pub = Publish{nullptr, nullptr, 0}) {
    loss_reduce(scratch, batch, reg, loss, loss_sum, pub);
}

inline Publish make_publish(const kgat_publish_t* p) {
    if (p == nullptr || p->serial_dev == nullptr || p->ring_host_mapped == nullptr || p->n_slots <= 0) return Publish{nullptr, nullptr, 0};
    return Publish{reinterpret_cast<unsigned long long*>(p->serial_dev), reinterpret_cast<volatile unsigned long long*>(p->ring_host_mapped),
                   p->n_slots};
}

// ---------------------------------------------------------------------------------------------
// BPR
// ---------------------------------------------------------------------------------------------
struct Tables {
    int n;
    int q[KGAT_MAX_LAYERS];  // float4 per row
    const float* p[KGAT_MAX_LAYERS];
    int64_t ld[KGAT_MAX_LAYERS];
};
struct GradTables {
    float* p[KGAT_MAX_LAYERS];
    int64_t ld[KGAT_MAX_LAYERS];
};

__global__ void __launch_bounds__(256) bpr_fwd_kernel(Tables T, const int64_t* __restrict__ users, const int64_t* __restrict__ pos,
                                                      const int64_t* __restrict__ neg, int batch, float* __restrict__ scratch) {
    const int lane = threadIdx.x & 31;
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= batch) return;
    const int64_t u = users[b], p = pos[b], n = neg[b];
    float sp = 0.f, sn = 0.f, l2 = 0.f;
    for (int t = 0; t < T.n; ++t) {
        for (int f = lane; f < T.q[t]; f += 32) {
            const float4 a = ldg4(T.p[t] + u * T.ld[t] + f * 4);
            const float4 x = ldg4(T.p[t] + p * T.ld[t] + f * 4);
            const float4 y = ldg4(T.p[t] + n * T.ld[t] + f * 4);
            sp += a.x * x.x + a.y * x.y + a.z * x.z + a.w * x.w;
            sn += a.x * y.x + a.y * y.y + a.z * y.z + a.w * y.w;
            l2 += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w + x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w + y.x * y.x +
                  y.y * y.y + y.z * y.z + y.w * y.w;
        }
    }
    sp = warp_sum(sp);
    sn = warp_sum(sn);
    l2 = warp_sum(l2);
    if (lane == 0) {
        scratch[b] = sp - sn;
        scratch[batch + b] = 0.5f * l2;
    }
}

__device__ __forceinline__ int64_t slot_id(const int64_t* __restrict__ a, const int64_t* __restrict__ b, const int64_t* __restrict__ c,
                                           int batch, int e) {
    return e < batch ? a[e] : (e < 2 * batch ? b[e - batch] : c[e - 2 * batch]);
}

// What the gradient of batch slot k (sample b = k mod B; role user / positive / negative) needs besides table rows: the sample's
// three ids and s = -d(-logsigmoid(m))/dm * g = sigmoid(-m) g
struct BprSlot {
    int64_t u, p, n;
    float s;
    int role;
};
__device__ __forceinline__ BprSlot bpr_slot(const int64_t* __restrict__ users, const int64_t* __restrict__ pos, const int64_t* __restrict__ neg,
                                            int batch, const float* __restrict__ scratch, float g, int k) {
    const int b = k % batch;
    return BprSlot{users[b], pos[b], neg[b], sigmoidf_(-scratch[b]) * g, k / batch};
}

// Contribution of one slot to its node's gradient, features [4f, 4f + 4); rounded as nvcc contracts
// acc += s (y - x) + lam a  (user),  -s a + lam x  (positive),  s a + lam y  (negative)
__device__ __forceinline__ void bpr_slot_add(const BprSlot& q, const float4& a, const float4& x, const float4& y, float lam, float4& acc) {
    if (q.role == 0) {
        acc.x = __fadd_rn(acc.x, __fmaf_rn(lam, a.x, __fmul_rn(q.s, __fsub_rn(y.x, x.x))));
        acc.y = __fadd_rn(acc.y, __fmaf_rn(lam, a.y, __fmul_rn(q.s, __fsub_rn(y.y, x.y))));
        acc.z = __fadd_rn(acc.z, __fmaf_rn(lam, a.z, __fmul_rn(q.s, __fsub_rn(y.z, x.z))));
        acc.w = __fadd_rn(acc.w, __fmaf_rn(lam, a.w, __fmul_rn(q.s, __fsub_rn(y.w, x.w))));
    } else if (q.role == 1) {
        acc.x = __fadd_rn(acc.x, __fmaf_rn(lam, x.x, __fmul_rn(-q.s, a.x)));
        acc.y = __fadd_rn(acc.y, __fmaf_rn(lam, x.y, __fmul_rn(-q.s, a.y)));
        acc.z = __fadd_rn(acc.z, __fmaf_rn(lam, x.z, __fmul_rn(-q.s, a.z)));
        acc.w = __fadd_rn(acc.w, __fmaf_rn(lam, x.w, __fmul_rn(-q.s, a.w)));
    } else {
        acc.x = __fadd_rn(acc.x, __fmaf_rn(lam, y.x, __fmul_rn(q.s, a.x)));
        acc.y = __fadd_rn(acc.y, __fmaf_rn(lam, y.y, __fmul_rn(q.s, a.y)));
        acc.z = __fadd_rn(acc.z, __fmaf_rn(lam, y.z, __fmul_rn(q.s, a.z)));
        acc.w = __fadd_rn(acc.w, __fmaf_rn(lam, y.w, __fmul_rn(q.s, a.w)));
    }
}

// One warp per id slot e of the batch (users, then positives, then negatives).  The warp of the FIRST slot holding a node
// sums the contributions of every slot holding it, in slot order, and adds the sum to the node's gradient row: a fixed
// summation order, so the gradients are bit-identical from run to run (float atomics would add in arrival order).  The block
// stages the slot ids in shared memory; one pass over them decides ownership and lists the node's slots (lane q keeps the
// q-th and its BprSlot), and the table rows of 4 slots are loaded at once.  A node held by more than 32 slots rescans the ids
// per feature chunk instead.
constexpr int kBprIdChunk = 2048;  // slot ids staged per pass (16 KB)
__global__ void __launch_bounds__(256) bpr_bwd_kernel(Tables T, GradTables G, const int64_t* __restrict__ users,
                                                      const int64_t* __restrict__ pos, const int64_t* __restrict__ neg, int batch,
                                                      float reg, const float* __restrict__ scratch,
                                                      const float* __restrict__ g_loss) {
    __shared__ int64_t s_ids[kBprIdChunk];
    const int lane = threadIdx.x & 31;
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int n3 = 3 * batch;
    const int64_t id = e < n3 ? slot_id(users, pos, neg, batch, e) : -1;
    bool owner = e < n3;
    int my_slot = -1, n_match = 0;
    for (int c0 = 0; c0 < n3; c0 += kBprIdChunk) {
        const int cn = n3 - c0 < kBprIdChunk ? n3 - c0 : kBprIdChunk;
        if (c0 > 0) __syncthreads();
        for (int t = threadIdx.x; t < cn; t += 256) s_ids[t] = slot_id(users, pos, neg, batch, c0 + t);
        __syncthreads();
        for (int k0 = c0; owner && k0 < c0 + cn; k0 += 32) {
            const int k = k0 + lane;
            const unsigned bal = __ballot_sync(kFull, k < c0 + cn && s_ids[k - c0] == id);
            const unsigned before = e - k0 >= 32 ? kFull : (e > k0 ? (1u << (e - k0)) - 1u : 0u);
            if (bal & before) owner = false;  // an earlier slot holds the node: its warp owns the row
            for (unsigned rest = bal; rest; rest &= rest - 1) {
                const int src = __ffs(rest) - 1;
                if (n_match + __popc(bal & ((1u << src) - 1u)) == lane) my_slot = k0 + src;
            }
            n_match += __popc(bal);
        }
    }
    if (!owner) return;
    const float g = g_loss[0] / (float)batch;
    const float lam = reg * g;
    BprSlot mine{0, 0, 0, 0.f, 0};
    if (my_slot >= 0) mine = bpr_slot(users, pos, neg, batch, scratch, g, my_slot);
    for (int t = 0; t < T.n; ++t) {
        if (G.p[t] == nullptr) continue;
        const float* tab = T.p[t];
        const int64_t ld = T.ld[t];
        for (int f = lane; f - lane < T.q[t]; f += 32) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n_match <= 32) {
                for (int q0 = 0; q0 < n_match; q0 += 4) {
                    BprSlot sl[4];
                    float4 a[4], x[4], y[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int src = q0 + u < n_match ? q0 + u : q0;
                        sl[u] = BprSlot{__shfl_sync(kFull, mine.u, src), __shfl_sync(kFull, mine.p, src), __shfl_sync(kFull, mine.n, src),
                                        __shfl_sync(kFull, mine.s, src), __shfl_sync(kFull, mine.role, src)};
                        if (f < T.q[t] && q0 + u < n_match) {
                            a[u] = ldg4(tab + sl[u].u * ld + f * 4);
                            x[u] = ldg4(tab + sl[u].p * ld + f * 4);
                            y[u] = ldg4(tab + sl[u].n * ld + f * 4);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (f < T.q[t] && q0 + u < n_match) bpr_slot_add(sl[u], a[u], x[u], y[u], lam, acc);
                }
            } else {
                for (int k0 = e; k0 < n3; k0 += 32) {
                    const int kk = k0 + lane;
                    unsigned hits = __ballot_sync(kFull, kk < n3 && slot_id(users, pos, neg, batch, kk) == id);
                    while (hits) {
                        const int k = k0 + __ffs(hits) - 1;
                        hits &= hits - 1;
                        if (f < T.q[t]) {
                            const BprSlot sl = bpr_slot(users, pos, neg, batch, scratch, g, k);
                            bpr_slot_add(sl, ldg4(tab + sl.u * ld + f * 4), ldg4(tab + sl.p * ld + f * 4), ldg4(tab + sl.n * ld + f * 4), lam, acc);
                        }
                    }
                }
            }
            if (f < T.q[t]) {
                float4* gp = reinterpret_cast<float4*>(G.p[t] + id * G.ld[t] + f * 4);
                float4 v = *gp;
                v.x += acc.x; v.y += acc.y; v.z += acc.z; v.w += acc.w;
                *gp = v;
            }
        }
    }
}

int pack_tables(const kgat_tables_t* t, Tables* out) {
    if (!t || t->n_tables <= 0 || t->n_tables > KGAT_MAX_LAYERS) return KGAT_ERR_INVALID_ARGUMENT;
    out->n = t->n_tables;
    for (int i = 0; i < t->n_tables; ++i) {
        if (t->dims[i] <= 0 || (t->dims[i] & 3) || (t->lds[i] & 3) || !t->tables[i]) return KGAT_ERR_INVALID_ARGUMENT;
        out->q[i] = t->dims[i] / 4;
        out->p[i] = t->tables[i];
        out->ld[i] = t->lds[i];
    }
    return KGAT_OK;
}

// ---------------------------------------------------------------------------------------------
// TransR:  x = e W_r  (row-vector convention).  One CTA of 4 warps per sample: the kernels are latency
// bound (512 samples, a 64-step dependent mat-vec each), so the rows j of W_r are split over the 4 warps
// and the partial projections are combined through shared memory.  Lane owns the KM consecutive output columns from KM * lane (ld_cols / red_cols).
// ---------------------------------------------------------------------------------------------
constexpr int kTrWarps = 4;

// A lane owns the KM CONSECUTIVE output columns [KM lane, KM lane + KM): its slice of a row of W_r / e_r is one 4 KM-byte load
// and its slice of a gradient row ONE vector reduction (red.global.add.v2/.v4.f32) -- the W_r gradient is 2.1 M scalar float
// atomics per 512-sample batch otherwise, which is what bounds the kernel.
template <int KM>
__device__ __forceinline__ void ld_cols(const float* __restrict__ p, int lane, float (&x)[KM]) {
    if constexpr (KM == 1) {
        x[0] = __ldg(p + lane);
    } else if constexpr (KM == 2) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(p) + lane);
        x[0] = v.x; x[1] = v.y;
    } else {
        static_assert(KM == 4, "KM is 1, 2 or 4");
        const float4 v = __ldg(reinterpret_cast<const float4*>(p) + lane);
        x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
    }
}
template <int KM>
__device__ __forceinline__ void red_cols(float* __restrict__ p, int lane, const float (&x)[KM]) {
    if constexpr (KM == 1) {
        atomicAdd(p + lane, x[0]);
    } else if constexpr (KM == 2) {
        asm volatile("red.relaxed.gpu.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p + 2 * lane), "f"(x[0]), "f"(x[1]) : "memory");
    } else {
        asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p + 4 * lane), "f"(x[0]), "f"(x[1]), "f"(x[2]), "f"(x[3])
                     : "memory");
    }
}

// partial projections of (e_h, e_p, e_n) over this warp's rows [j0, j0 + JW) of W_r
template <int D, int KM>
__device__ __forceinline__ void transr_partial(const float* __restrict__ Wr, const float* __restrict__ emb, int64_t h, int64_t p, int64_t n,
                                               int warp, int lane, float& eh, float& ep, float& en, float (&xh)[KM], float (&xp)[KM],
                                               float (&xn)[KM]) {
    constexpr int K = KM * 32;
    constexpr int JW = D / kTrWarps;  // rows of W_r per warp (8, 16 or 32)
    const int j0 = warp * JW;
    eh = ep = en = 0.f;
    if (lane < JW) {
        eh = __ldg(emb + h * D + j0 + lane);
        ep = __ldg(emb + p * D + j0 + lane);
        en = __ldg(emb + n * D + j0 + lane);
    }
#pragma unroll
    for (int m = 0; m < KM; ++m) xh[m] = xp[m] = xn[m] = 0.f;
#pragma unroll 8
    for (int jj = 0; jj < JW; ++jj) {
        const float a = __shfl_sync(kFull, eh, jj);
        const float b = __shfl_sync(kFull, ep, jj);
        const float c = __shfl_sync(kFull, en, jj);
        float w[KM];
        ld_cols<KM>(Wr + (j0 + jj) * K, lane, w);
#pragma unroll
        for (int m = 0; m < KM; ++m) {
            xh[m] = fmaf(a, w[m], xh[m]);
            xp[m] = fmaf(b, w[m], xp[m]);
            xn[m] = fmaf(c, w[m], xn[m]);
        }
    }
}

// combine the 4 warps' partials: every warp returns with the full projections
template <int KM>
__device__ __forceinline__ void transr_combine(float (*part)[3][KM * 32], int warp, int lane, float (&xh)[KM], float (&xp)[KM],
                                               float (&xn)[KM]) {
#pragma unroll
    for (int m = 0; m < KM; ++m) {
        part[warp][0][lane + 32 * m] = xh[m];
        part[warp][1][lane + 32 * m] = xp[m];
        part[warp][2][lane + 32 * m] = xn[m];
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < KM; ++m) {
        float a = 0.f, b = 0.f, c = 0.f;
#pragma unroll
        for (int w = 0; w < kTrWarps; ++w) {
            a += part[w][0][lane + 32 * m];
            b += part[w][1][lane + 32 * m];
            c += part[w][2][lane + 32 * m];
        }
        xh[m] = a;
        xp[m] = b;
        xn[m] = c;
    }
}

template <int DM, int KM>
__global__ void __launch_bounds__(128) transr_fwd_kernel(const float* __restrict__ emb, const float* __restrict__ rel_emb,
                                                         const float* __restrict__ W, const int64_t* __restrict__ heads,
                                                         const int64_t* __restrict__ rels, const int64_t* __restrict__ pt,
                                                         const int64_t* __restrict__ nt, int batch, float* __restrict__ scratch) {
    constexpr int D = DM * 32, K = KM * 32;
    __shared__ float part[kTrWarps][3][K];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x;
    const int64_t h = heads[b], r = rels[b], p = pt[b], n = nt[b];
    float eh, ep, en, xh[KM], xp[KM], xn[KM];
    transr_partial<D, KM>(W + r * (int64_t)D * K, emb, h, p, n, warp, lane, eh, ep, en, xh, xp, xn);
    transr_combine<KM>(part, warp, lane, xh, xp, xn);
    if (warp != 0) return;
    float ps = 0.f, ns = 0.f, l2 = 0.f;
    float er[KM];
    ld_cols<KM>(rel_emb + r * K, lane, er);
#pragma unroll
    for (int m = 0; m < KM; ++m) {
        const float dp = xh[m] + er[m] - xp[m];
        const float dn = xh[m] + er[m] - xn[m];
        ps = fmaf(dp, dp, ps);
        ns = fmaf(dn, dn, ns);
        l2 += xh[m] * xh[m] + er[m] * er[m] + xp[m] * xp[m] + xn[m] * xn[m];
    }
    ps = warp_sum(ps);
    ns = warp_sum(ns);
    l2 = warp_sum(l2);
    if (lane == 0) {
        scratch[b] = ns - ps;
        scratch[batch + b] = 0.5f * l2;
    }
}

// FUSED: forward and backward in one pass (the backward recomputes the projections anyway): the kernel derives the
// sample's margin itself, records it (and the L2 term) in `scratch` for the loss reduction that follows, and uses
// d loss / d batch-loss = 1.
template <int DM, int KM, bool FUSED = false>
__global__ void __launch_bounds__(128) transr_bwd_kernel(const float* __restrict__ emb, const float* __restrict__ rel_emb,
                                                         const float* __restrict__ W, const int64_t* __restrict__ heads,
                                                         const int64_t* __restrict__ rels, const int64_t* __restrict__ pt,
                                                         const int64_t* __restrict__ nt, int batch, float reg,
                                                         float* __restrict__ scratch, const float* __restrict__ g_loss,
                                                         float* __restrict__ g_emb, float* __restrict__ g_rel,
                                                         float* __restrict__ g_W, const int32_t* __restrict__ row_slot,
                                                         float* __restrict__ work = nullptr) {
    // work != nullptr: no atomics -- the sample's projection gradients go to work[b] (g_xh, g_xp, g_xn, g_er; K each) and its
    // embedding gradients to its own compact rows b, B + b, 2B + b of g_emb; transr_reduce_kernel sums both in sample order
    constexpr int D = DM * 32, K = KM * 32;
    constexpr int JW = D / kTrWarps;
    __shared__ float part[kTrWarps][3][K];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x;
    const int64_t h = heads[b], r = rels[b], p = pt[b], n = nt[b];
    const float* Wr = W + r * (int64_t)D * K;
    float eh, ep, en, xh[KM], xp[KM], xn[KM];
    transr_partial<D, KM>(Wr, emb, h, p, n, warp, lane, eh, ep, en, xh, xp, xn);
    transr_combine<KM>(part, warp, lane, xh, xp, xn);

    float er[KM];
    ld_cols<KM>(rel_emb + r * K, lane, er);
    float margin;
    if (FUSED) {
        float ps = 0.f, ns = 0.f, l2 = 0.f;
#pragma unroll
        for (int m = 0; m < KM; ++m) {
            const float dp = xh[m] + er[m] - xp[m];
            const float dn = xh[m] + er[m] - xn[m];
            ps = fmaf(dp, dp, ps);
            ns = fmaf(dn, dn, ns);
            l2 += xh[m] * xh[m] + er[m] * er[m] + xp[m] * xp[m] + xn[m] * xn[m];
        }
        ps = warp_sum(ps);
        ns = warp_sum(ns);
        l2 = warp_sum(l2);
        margin = ns - ps;
        if (warp == 0 && lane == 0) {
            scratch[b] = margin;
            scratch[batch + b] = 0.5f * l2;
        }
    } else {
        margin = scratch[b];
    }
    const float g = (FUSED ? 1.f : g_loss[0]) / (float)batch;
    const float s2 = 2.f * sigmoidf_(-margin) * g;  // loss = -logsigmoid(ns - ps)
    const float lam = reg * g;
    float gxh[KM], gxp[KM], gxn[KM], ger[KM];
#pragma unroll
    for (int m = 0; m < KM; ++m) {
        const float dp = xh[m] + er[m] - xp[m];
        const float dn = xh[m] + er[m] - xn[m];
        const float gdp = s2 * dp;   // dL/d dpos
        const float gdn = -s2 * dn;  // dL/d dneg
        gxh[m] = gdp + gdn + lam * xh[m];
        gxp[m] = -gdp + lam * xp[m];
        gxn[m] = -gdn + lam * xn[m];
        ger[m] = gdp + gdn + lam * er[m];
    }
    if (work != nullptr) {
        if (warp == 0) {
            float* wb = work + (int64_t)b * 4 * K + KM * lane;
#pragma unroll
            for (int m = 0; m < KM; ++m) {
                wb[m] = gxh[m];
                wb[K + m] = gxp[m];
                wb[2 * K + m] = gxn[m];
                wb[3 * K + m] = ger[m];
            }
        }
    } else if (warp == 0) {
        red_cols<KM>(g_rel + r * K, lane, ger);
    }
    // this warp's rows of W_r: d e[j] = <g_x, W_r[j, :]>, d W_r[j, :] += e[j] * g_x
    const int j0 = warp * JW;
    float* gWr = g_W + r * (int64_t)D * K;
    float geh = 0.f, gep = 0.f, gen = 0.f;
#pragma unroll 4
    for (int jj = 0; jj < JW; ++jj) {
        const int j = j0 + jj;
        const float a = __shfl_sync(kFull, eh, jj);
        const float bb = __shfl_sync(kFull, ep, jj);
        const float c = __shfl_sync(kFull, en, jj);
        float ph = 0.f, pp = 0.f, pn = 0.f;
        float w[KM], gw[KM];
        ld_cols<KM>(Wr + j * K, lane, w);
#pragma unroll
        for (int m = 0; m < KM; ++m) {
            ph = fmaf(gxh[m], w[m], ph);
            pp = fmaf(gxp[m], w[m], pp);
            pn = fmaf(gxn[m], w[m], pn);
            gw[m] = a * gxh[m] + bb * gxp[m] + c * gxn[m];
        }
        if (work == nullptr) red_cols<KM>(gWr + j * K, lane, gw);
        ph = warp_sum(ph);
        pp = warp_sum(pp);
        pn = warp_sum(pn);
        if (lane == jj) {
            geh = ph;
            gep = pp;
            gen = pn;
        }
    }
    if (lane < JW && work != nullptr) {
        g_emb[(int64_t)b * D + j0 + lane] = geh;
        g_emb[(int64_t)(batch + b) * D + j0 + lane] = gep;
        g_emb[(int64_t)(2 * batch + b) * D + j0 + lane] = gen;
    } else if (lane < JW) {
        // dense gradient table indexed by node, or compact rows indexed through row_slot (kgat_transr_claim_rows)
        const int64_t gh = row_slot ? row_slot[h] : h, gp = row_slot ? row_slot[p] : p, gn = row_slot ? row_slot[n] : n;
        atomicAdd(g_emb + gh * D + j0 + lane, geh);
        atomicAdd(g_emb + gp * D + j0 + lane, gep);
        atomicAdd(g_emb + gn * D + j0 + lane, gen);
    }
}

// Second pass of the deterministic TransR backward (transr_bwd_kernel with `work`), every sum in a fixed order:
//  * blocks [0, B * D / JB): block (b, jb) -- if sample b is the first of its relation r -- adds the relation's samples' outer
//    products e^T g_x to rows [JB jb, JB jb + JB) of g_W[r], and block (b, 0) their g_er to g_rel[r].  Warp w takes the samples
//    i = b + w (mod kRdWarps) in increasing order; the warps' partial sums are combined in warp order;
//  * the next blocks: one warp per id slot e; the slot that owns its node's compact row (row_slot[node] == e) replaces that
//    row by the sum of the rows of every slot holding the node, in slot order;
//  * with `loss` set, one last block reduces the loss (loss_reduce): the margins are complete before this launch starts.
// A warp copies the slices of its next kTrStage<KM> samples into shared memory with cp.async, all in flight at once, before
// it adds any of them; the id slots are staged in shared memory once per block, and a node's gradient rows are read 4 at a
// time.  Measured on a B200 at d = 64, B = 512, this takes 5-6 us off the launch when the relations are spread out, but
// not when one relation holds most of the batch: its 4 blocks take as long as before, so load latency is not their bound.
constexpr int kRdWarps = 8;
// rows of g_W[r] per block: the warps' partial sums of the block's JB x K tile plus g_er stay inside 48 KB of shared memory
__host__ __device__ constexpr int transr_reduce_rows(int d) { return d >= 128 ? 8 : 16; }
// samples a warp stages at once: the block's staging buffers stay inside 48 KB of shared memory
template <int KM>
constexpr int kTrStage = KM == 4 ? 2 : (KM == 2 ? 4 : 8);

__device__ __forceinline__ void cp_async16(float* dst, const float* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
// `work` starts 2B floats into the scratch, so its rows are only 8-byte aligned
__device__ __forceinline__ void cp_async8(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory"); }

template <int DM, int KM>
__global__ void __launch_bounds__(kRdWarps * 32, DM == 1 ? 4 : 3) transr_reduce_kernel(const float* __restrict__ emb, const int64_t* __restrict__ heads,
                                                                     const int64_t* __restrict__ rels, const int64_t* __restrict__ pt,
                                                                     const int64_t* __restrict__ nt, int batch, const float* __restrict__ work,
                                                                     const int32_t* __restrict__ row_slot, float* __restrict__ g_rows,
                                                                     float* __restrict__ g_rel, float* __restrict__ g_W,
                                                                     const float* __restrict__ scratch = nullptr, float reg = 0.f,
                                                                     float* __restrict__ loss = nullptr, float* __restrict__ loss_sum = nullptr,
                                                                     Publish pub = Publish{nullptr, nullptr, 0}) {
    constexpr int D = DM * 32, K = KM * 32, JB = transr_reduce_rows(DM * 32), NJB = D / JB, NOUT = JB * K + K;
    constexpr int S = kTrStage<KM>, SF = 3 * JB + 4 * K;  // per staged sample: e_h, e_p, e_n rows [j0, j0 + JB), then work row
    constexpr int NBUF = kRdWarps * NOUT > kRdWarps * S * SF ? kRdWarps * NOUT : kRdWarps * S * SF;
    // staging buffers, then the warps' partial sums (relation blocks); the id slots (row blocks)
    __shared__ __align__(16) float s_buf[NBUF];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int blk = blockIdx.x;
    if (blk < batch * NJB) {
        const int b = blk / NJB, jb = blk % NJB, j0 = jb * JB;
        const int64_t r = rels[b];
        int dup = 0;
        for (int i = tid; i < b; i += kRdWarps * 32) dup |= rels[i] == r;
        if (__syncthreads_or(dup)) return;
        float acc[JB][KM], acc_r[KM];
#pragma unroll
        for (int m = 0; m < KM; ++m) {
            acc_r[m] = 0.f;
#pragma unroll
            for (int jj = 0; jj < JB; ++jj) acc[jj][m] = 0.f;
        }
        float* stage = s_buf + warp * S * SF;
        const int nw2 = (jb == 0 ? 4 : 3) * K / 2;  // 8-byte pieces of a work row this block reads (g_er only in block jb = 0)
        for (int base = b + warp; base < batch; base += kRdWarps * 32) {
            const int il = base + kRdWarps * lane;
            const bool mine = il < batch && rels[il] == r;
            long long hl = 0, pl = 0, nl = 0;
            if (mine) {
                hl = heads[il];
                pl = pt[il];
                nl = nt[il];
            }
            unsigned hits = __ballot_sync(kFull, mine);
            while (hits) {
                unsigned chunk = hits;  // the warp's next S samples, in increasing order
                for (int q = 0; q < S && hits; ++q) hits &= hits - 1;
                chunk &= ~hits;
                int q = 0;
                for (unsigned rest = chunk; rest; rest &= rest - 1, ++q) {
                    const int src = __ffs(rest) - 1;
                    const long long h = __shfl_sync(kFull, hl, src), p = __shfl_sync(kFull, pl, src), n = __shfl_sync(kFull, nl, src);
                    float* st = stage + q * SF;
                    if (lane < 3 * JB / 4) {
                        const int row = lane / (JB / 4), c = 4 * (lane % (JB / 4));
                        cp_async16(st + row * JB + c, emb + (row == 0 ? h : (row == 1 ? p : n)) * D + j0 + c);
                    }
                    const float* wi = work + (int64_t)(base + kRdWarps * src) * 4 * K;
                    for (int c = lane; c < nw2; c += 32) cp_async8(st + 3 * JB + 2 * c, wi + 2 * c);
                }
                cp_async_wait_all();
                __syncwarp();
                for (int qq = 0; qq < q; ++qq) {
                    const float* ev = stage + qq * SF;
                    const float* gv = ev + 3 * JB + KM * lane;
#pragma unroll
                    for (int m = 0; m < KM; ++m) {
                        const float gh = gv[m], gp = gv[K + m], gn = gv[2 * K + m];
                        // acc += eh gh + ep gp + en gn, rounded as nvcc contracts it: fma(en, gn, fma(eh, gh, ep gp))
#pragma unroll
                        for (int jj = 0; jj < JB; ++jj)
                            acc[jj][m] = __fadd_rn(acc[jj][m], __fmaf_rn(ev[2 * JB + jj], gn, __fmaf_rn(ev[jj], gh, __fmul_rn(ev[JB + jj], gp))));
                        if (jb == 0) acc_r[m] += gv[3 * K + m];
                    }
                }
                __syncwarp();  // the stage is refilled next
            }
        }
        __syncthreads();  // s_part overlays the other warps' stages
        float (*s_part)[NOUT] = reinterpret_cast<float (*)[NOUT]>(s_buf);
#pragma unroll
        for (int m = 0; m < KM; ++m) {
#pragma unroll
            for (int jj = 0; jj < JB; ++jj) s_part[warp][jj * K + KM * lane + m] = acc[jj][m];
            s_part[warp][JB * K + KM * lane + m] = acc_r[m];
        }
        __syncthreads();
        float* gWr = g_W + r * (int64_t)D * K;
        for (int o = tid; o < NOUT; o += kRdWarps * 32) {
            float sum = 0.f;
#pragma unroll
            for (int w = 0; w < kRdWarps; ++w) sum += s_part[w][o];
            if (o < JB * K) gWr[(int64_t)(j0 + o / K) * K + o % K] += sum;
            else if (jb == 0) g_rel[r * K + (o - JB * K)] += sum;
        }
        return;
    }
    blk -= batch * NJB;
    const int n3 = 3 * batch;
    if (blk * kRdWarps >= n3) {
        loss_reduce(scratch, batch, reg, loss, loss_sum, pub);
        return;
    }
    const int e = blk * kRdWarps + warp;
    const int64_t id = e < n3 ? slot_id(heads, pt, nt, batch, e) : -1;
    const bool owner = e < n3 && row_slot[id] == e;
    constexpr int CH = NBUF * 4 / 8;  // id slots per staged chunk
    int64_t* s_ids = reinterpret_cast<int64_t*>(s_buf);
    float acc[DM];
#pragma unroll
    for (int c = 0; c < DM; ++c) acc[c] = 0.f;
    for (int c0 = 0; c0 < n3; c0 += CH) {
        const int cn = n3 - c0 < CH ? n3 - c0 : CH;
        if (c0 > 0) __syncthreads();
        for (int t = tid; t < cn; t += kRdWarps * 32) s_ids[t] = slot_id(heads, pt, nt, batch, c0 + t);
        __syncthreads();
        if (!owner) continue;
        for (int k0 = 0; k0 < cn; k0 += 32) {
            unsigned hits = __ballot_sync(kFull, k0 + lane < cn && s_ids[k0 + lane] == id);
            while (hits) {
                int ks[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    ks[q] = hits ? c0 + k0 + __ffs(hits) - 1 : -1;
                    hits &= hits - 1;
                }
                float v[4][DM];
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int c = 0; c < DM; ++c) v[q][c] = ks[q] >= 0 ? g_rows[(int64_t)ks[q] * D + lane + 32 * c] : 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (ks[q] >= 0) {
#pragma unroll
                        for (int c = 0; c < DM; ++c) acc[c] += v[q][c];
                    }
            }
        }
    }
    if (!owner) return;
#pragma unroll
    for (int c = 0; c < DM; ++c) g_rows[(int64_t)e * D + lane + 32 * c] = acc[c];
}

// Compact gradient rows for the embedding table: the 3B ids of a batch claim a slot per DISTINCT node
// (row_slot[node] = index of the first claimant, -1 = untouched; the Adam kernel resets the claims), and the
// 3B x d gradient rows are zeroed -- instead of zeroing and re-reading an n_nodes x d gradient table per step.
__global__ void transr_claim_rows_kernel(const int64_t* __restrict__ heads, const int64_t* __restrict__ pt, const int64_t* __restrict__ nt,
                                         int batch, int d, int32_t* __restrict__ row_slot, float4* __restrict__ g_rows,
                                         float4* __restrict__ zero_a = nullptr, int n_a = 0, float4* __restrict__ zero_b = nullptr,
                                         int n_b = 0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 3 * batch * (d / 4)) g_rows[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n_a) zero_a[i] = make_float4(0.f, 0.f, 0.f, 0.f);  // the step's other gradient buffers, zeroed in the same launch
    if (i < n_b) zero_b[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < 3 * batch) {
        const int64_t id = i < batch ? heads[i] : (i < 2 * batch ? pt[i - batch] : nt[i - 2 * batch]);
        atomicCAS(row_slot + id, -1, i);
    }
}

// T[ids[i], :] = 0: re-zero the few rows a sparse scatter touched instead of memsetting the whole table
__global__ void zero_rows_i64_kernel(float* __restrict__ T, int64_t ld, int d4, const int64_t* __restrict__ ids, int64_t n_ids,
                                     int64_t n_rows) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_ids * d4) return;
    const int64_t r = ids[i / d4];
    if (r < 0 || r >= n_rows) return;
    reinterpret_cast<float4*>(T + r * ld)[i % d4] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// dense[id, :] = g_rows[slot, :] for every batch id whose claim this entry won (row_slot[id] == its index): the dense
// embedding gradient autograd would hand out, restricted to the <= 3B rows that are not zero
__global__ void transr_rows_to_dense_kernel(const float4* __restrict__ g_rows, const int32_t* __restrict__ row_slot,
                                            const int64_t* __restrict__ heads, const int64_t* __restrict__ pt, const int64_t* __restrict__ nt,
                                            int batch, int d4, float* __restrict__ dense, int64_t ld, int64_t* __restrict__ keep_h,
                                            int64_t* __restrict__ keep_pt, int64_t* __restrict__ keep_nt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3 * batch * d4) return;
    const int e = i / d4, q = i % d4;
    const int64_t id = e < batch ? heads[e] : (e < 2 * batch ? pt[e - batch] : nt[e - 2 * batch]);
    if (keep_h != nullptr && q == 0) {  // remember whose rows the dense view now holds (cleared before the next batch's rows go in)
        if (e < batch) keep_h[e] = id;
        else if (e < 2 * batch) keep_pt[e - batch] = id;
        else keep_nt[e - 2 * batch] = id;
    }
    if (row_slot[id] != e) return;
    reinterpret_cast<float4*>(dense + id * ld)[q] = g_rows[(int64_t)e * d4 + q];
}

// dense[ids[i], :] = 0 and row_slot[ids[i]] = -1: undo what the previous batch left behind
__global__ void transr_release_rows_kernel(float* __restrict__ dense, int64_t ld, int d4, const int64_t* __restrict__ ids, int64_t n_ids,
                                           int64_t n_rows, int32_t* __restrict__ row_slot) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_ids * d4) return;
    const int64_t r = ids[i / d4];
    if (r < 0 || r >= n_rows) return;
    reinterpret_cast<float4*>(dense + r * ld)[i % d4] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i % d4 == 0) row_slot[r] = -1;
}

}  // namespace
}  // namespace kgat

using namespace kgat;

extern "C" {

int kgat_transr_rows_to_dense(const float* g_rows, const int32_t* row_slot, const int64_t* heads, const int64_t* pos_tails,
                              const int64_t* neg_tails, int32_t batch, int32_t d, float* dense, int64_t ld, int64_t* keep_heads,
                              int64_t* keep_pos_tails, int64_t* keep_neg_tails, void* stream) {
    if ((keep_heads != nullptr) != (keep_pos_tails != nullptr) || (keep_heads != nullptr) != (keep_neg_tails != nullptr)) return KGAT_ERR_INVALID_ARGUMENT;
    if (!g_rows || !row_slot || !heads || !pos_tails || !neg_tails || !dense || batch <= 0 || d <= 0 || (d & 3) || (ld & 3))
        return KGAT_ERR_INVALID_ARGUMENT;
    const int total = 3 * batch * (d / 4);
    transr_rows_to_dense_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(g_rows), row_slot, heads,
                                                                                    pos_tails, neg_tails, batch, d / 4, dense, ld, keep_heads,
                                                                                    keep_pos_tails, keep_neg_tails);
    return check_launch();
}

int kgat_transr_release_rows(float* dense, int64_t n_rows, int64_t ld, int32_t d, const int64_t* ids64, int64_t n_ids, int32_t* row_slot,
                             void* stream) {
    if (!dense || !ids64 || !row_slot || n_rows <= 0 || d <= 0 || (d & 3) || (ld & 3) || n_ids < 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_ids == 0) return KGAT_OK;
    const int64_t total = n_ids * (d / 4);
    transr_release_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dense, ld, d / 4, ids64, n_ids, n_rows, row_slot);
    return check_launch();
}

int kgat_zero_rows_i64(float* T, int64_t n_rows, int64_t ld, int32_t d, const int64_t* ids64, int64_t n_ids, void* stream) {
    if (!T || !ids64 || n_rows <= 0 || d <= 0 || (d & 3) || (ld & 3) || n_ids < 0) return KGAT_ERR_INVALID_ARGUMENT;
    if (n_ids == 0) return KGAT_OK;
    const int64_t total = n_ids * (d / 4);
    zero_rows_i64_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(T, ld, d / 4, ids64, n_ids, n_rows);
    return check_launch();
}

int kgat_bpr_forward(const kgat_tables_t* tables, const int64_t* users, const int64_t* pos, const int64_t* neg, int32_t batch,
                     float reg, float* loss, float* loss_sum, float* margin, const kgat_publish_t* publish, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    Tables T;
    int rc = pack_tables(tables, &T);
    if (rc != KGAT_OK) return rc;
    if (batch <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    bpr_fwd_kernel<<<(batch * 32 + 255) / 256, 256, 0, stream>>>(T, users, pos, neg, batch, margin);
    loss_reduce_kernel<<<1, 256, 0, stream>>>(margin, batch, reg, loss, loss_sum, make_publish(publish));
    return check_launch();
}

int kgat_bpr_backward(const kgat_tables_t* tables, const kgat_grad_tables_t* grads, const int64_t* users, const int64_t* pos,
                      const int64_t* neg, int32_t batch, float reg, const float* margin, const float* g_loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    Tables T;
    int rc = pack_tables(tables, &T);
    if (rc != KGAT_OK) return rc;
    if (batch <= 0 || !grads || grads->n_tables != tables->n_tables) return KGAT_ERR_INVALID_ARGUMENT;
    GradTables G;
    for (int i = 0; i < T.n; ++i) {
        if (grads->tables[i] && (grads->dims[i] != tables->dims[i] || (grads->lds[i] & 3))) return KGAT_ERR_INVALID_ARGUMENT;
        G.p[i] = grads->tables[i];
        G.ld[i] = grads->lds[i];
    }
    bpr_bwd_kernel<<<(3 * batch * 32 + 255) / 256, 256, 0, stream>>>(T, G, users, pos, neg, batch, reg, margin, g_loss);
    return check_launch();
}

#define KGAT_TRANSR_DISPATCH(CALL)                                            \
    if (d == 32 && k == 32) { constexpr int DM = 1, KM = 1; CALL; }           \
    else if (d == 64 && k == 64) { constexpr int DM = 2, KM = 2; CALL; }      \
    else if (d == 128 && k == 128) { constexpr int DM = 4, KM = 4; CALL; }    \
    else return KGAT_ERR_UNSUPPORTED;

int kgat_transr_forward(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k, const int64_t* heads,
                        const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, float reg, float* loss,
                        float* margin, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (batch <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    const unsigned blocks = (unsigned)batch;  // one 4-warp CTA per sample
    KGAT_TRANSR_DISPATCH((transr_fwd_kernel<DM, KM><<<blocks, 128, 0, stream>>>(emb, rel_emb, W, heads, rels, pos_tails, neg_tails,
                                                                               batch, margin)));
    loss_reduce_kernel<<<1, 256, 0, stream>>>(margin, batch, reg, loss);
    return check_launch();
}

int kgat_transr_backward(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k, const int64_t* heads,
                         const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, float reg,
                         const float* margin, const float* g_loss, float* g_emb, float* g_rel_emb, float* g_W, const int32_t* row_slot,
                         void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (batch <= 0) return KGAT_ERR_INVALID_ARGUMENT;
    const unsigned blocks = (unsigned)batch;  // one 4-warp CTA per sample
    KGAT_TRANSR_DISPATCH((transr_bwd_kernel<DM, KM><<<blocks, 128, 0, stream>>>(emb, rel_emb, W, heads, rels, pos_tails, neg_tails,
                                                                               batch, reg, const_cast<float*>(margin), g_loss, g_emb,
                                                                               g_rel_emb, g_W, row_slot)));
    return check_launch();
}

int kgat_transr_step(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k, int32_t n_rel, const int64_t* heads,
                     const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, float reg, float* loss,
                     float* loss_sum, float* margin, int32_t* row_slot, float* g_rows, float* g_rel_emb, float* g_W,
                     const kgat_publish_t* publish, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (batch <= 0 || d <= 0 || (d & 3) || (k & 3) || n_rel <= 0 || !row_slot || !g_rows || !g_rel_emb || !g_W || !loss || !margin)
        return KGAT_ERR_INVALID_ARGUMENT;
    const int n_rows4 = 3 * batch * (d / 4), n_rel4 = n_rel * k / 4, n_w4 = n_rel * d * (k / 4);
    const int n = n_rows4 > n_w4 ? (n_rows4 > n_rel4 ? n_rows4 : n_rel4) : (n_w4 > n_rel4 ? n_w4 : n_rel4);
    transr_claim_rows_kernel<<<(n + 255) / 256, 256, 0, stream>>>(heads, pos_tails, neg_tails, batch, d, row_slot,
                                                                 reinterpret_cast<float4*>(g_rows), reinterpret_cast<float4*>(g_rel_emb),
                                                                 n_rel4, reinterpret_cast<float4*>(g_W), n_w4);
    const unsigned blocks = (unsigned)batch;
    // margin[0, 2B): per-sample margin and L2 term; margin[2B, 2B + 4BK): the deterministic backward's work rows
    float* work = margin + 2 * batch;
    // relation blocks, row blocks, one loss block
    const unsigned reduce_blocks = (unsigned)(batch * (d / transr_reduce_rows(d)) + (3 * batch + kRdWarps - 1) / kRdWarps + 1);
    KGAT_TRANSR_DISPATCH((transr_bwd_kernel<DM, KM, true><<<blocks, 128, 0, stream>>>(emb, rel_emb, W, heads, rels, pos_tails, neg_tails,
                                                                                     batch, reg, margin, nullptr, g_rows, g_rel_emb, g_W,
                                                                                     row_slot, work),
                          transr_reduce_kernel<DM, KM><<<reduce_blocks, kRdWarps * 32, 0, stream>>>(emb, heads, rels, pos_tails, neg_tails, batch, work,
                                                                                          row_slot, g_rows, g_rel_emb, g_W, margin, reg, loss,
                                                                                          loss_sum, make_publish(publish))));
    return check_launch();
}

/* kgat_transr_step without its first launch: the compact rows were claimed and the gradient buffers zeroed by the caller
 * (kgat_adam_rolling_prepare does both while it brings the batch rows up to date) */
int kgat_transr_step_claimed(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k, const int64_t* heads,
                             const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, float reg, float* loss,
                             float* loss_sum, float* margin, const int32_t* row_slot, float* g_rows, float* g_rel_emb, float* g_W,
                             const kgat_publish_t* publish, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (batch <= 0 || d <= 0 || !row_slot || !g_rows || !g_rel_emb || !g_W || !loss || !margin) return KGAT_ERR_INVALID_ARGUMENT;
    const unsigned blocks = (unsigned)batch;
    // margin[0, 2B): per-sample margin and L2 term; margin[2B, 2B + 4BK): the deterministic backward's work rows
    float* work = margin + 2 * batch;
    // relation blocks, row blocks, one loss block
    const unsigned reduce_blocks = (unsigned)(batch * (d / transr_reduce_rows(d)) + (3 * batch + kRdWarps - 1) / kRdWarps + 1);
    KGAT_TRANSR_DISPATCH((transr_bwd_kernel<DM, KM, true><<<blocks, 128, 0, stream>>>(emb, rel_emb, W, heads, rels, pos_tails, neg_tails,
                                                                                     batch, reg, margin, nullptr, g_rows, g_rel_emb, g_W,
                                                                                     row_slot, work),
                          transr_reduce_kernel<DM, KM><<<reduce_blocks, kRdWarps * 32, 0, stream>>>(emb, heads, rels, pos_tails, neg_tails, batch, work,
                                                                                          row_slot, g_rows, g_rel_emb, g_W, margin, reg, loss,
                                                                                          loss_sum, make_publish(publish))));
    return check_launch();
}

int kgat_transr_claim_rows(const int64_t* heads, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, int32_t d,
                           int32_t* row_slot, float* g_rows, void* stream_) {
    if (batch <= 0 || d <= 0 || (d & 3) || !row_slot || !g_rows) return KGAT_ERR_INVALID_ARGUMENT;
    const int n = 3 * batch * (d / 4);
    transr_claim_rows_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream_>>>(heads, pos_tails, neg_tails, batch, d, row_slot,
                                                                              reinterpret_cast<float4*>(g_rows));
    return check_launch();
}

}  // extern "C"
