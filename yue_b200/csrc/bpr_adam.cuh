// K10: BPR's shipped training -- replaces the TF-1 graph and loop of recommender/cf/BPR.py:65-129 (SURVEY.md 3.3, row a10):
// per step, `batch` training events drawn uniformly with replacement (next_batch, 65-81), `negatives` unplayed tracks per
// event, the softplus BPR loss over the batch x negatives triplets with regU on all three rows (93-115) and one AdamOptimizer
// step on EVERY row of U and V per iteration of the loop (121-129).
//
//   x = U_u . V_i - U_u . V_j      loss = sum softplus(-x) + reg/2 (|U_u|^2 + |V_i|^2 + |V_j|^2)       (rows read before the step)
//   c = 1 - sigmoid(x):   dU_u = -c (V_i - V_j) + reg U_u,   dV_i = -c U_u + reg V_i,   dV_j = c U_u + reg V_j
//   Adam: m = 0.9 m + 0.1 g,  v = 0.999 v + 0.001 g^2,  var -= lr_t m / (sqrt(v) + 1e-8),  lr_t from the host per step
//
// Sampler (Philox stream of K1, oracle/philox.py): row b of step s draws its event with (epoch s, event b, slot 4095,
// attempt 0) over T instead of n, e = (r T) >> 32; negative k of the row is slot k with the usual rejection against the
// user's play row.  The batch is a pure function of (seed, s).
//
// B200 shape.  A step is five short phases and one streaming pass, each its own launch on the handle's stream:
//   triplet   a group of G lanes per TRIPLET (51 200 of them at the reference's 512 x 100; 512 rows would fill 3.5 warps per
//             SM): draws, three row loads, loss and c; counts the triplet's graph rows (slots) per row with an atomic
//   row       a group per batch row: the user's gradient summed over its negatives in k order, C_b = sum_k c, a copy of U_u
//   alloc / scatter / rank    per slot: every touched row gets a bucket of its slots; the buckets are then ordered by
//             slot id, so every row's contributions are added in one fixed order (same bits on every run, whoever
//             won the atomics)
//   adam      every float4 of U and V: the row's gradient from its bucket (touched rows only), Adam's step; the dense pass
//             streams var, m and v in and out, 6 (m + n) ld 4 bytes, which is what bounds a step at config C2's shape
// Slots: [0, B) the rows' users (contribution: the row's user gradient), [B, 2B) the rows' positives (-C_b U_u + K reg V_i),
// [2B, 2B + B K) the negatives (c U_u + reg V_j).  U_u comes from the copy the row phase took: the adam pass rewrites U.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "lightgcn.cuh"     // GcnVec, gcn_group_sum, gcn_group_mask: the lane-group row arithmetic of K9
#include "philox.cuh"

namespace yue {

constexpr uint32_t kBprAdamPosSlot = 4095;   // the positive's Philox slot; negatives use slots 0 .. K-1 (K <= 4095)
constexpr int kBprAdamThreads = 256;

struct BprAdamParams {
    int64_t m, n, T;
    int ld, B, K;                                  // row stride; batch rows, negatives per row
    const int32_t* ev_user;                        // [T] user of every event (the event CSR's rows)
    const int32_t* ev_items;                       // [T] device copy: hot positives are -slot-1 (SgdParams::hot_items)
    const int32_t* hot_items;
    const int64_t* uq_indptr; const int32_t* uq_items;
    float* P; float* Q; float* am; float* av;      // tables; Adam's moments [m + n, ld], users first
    const int32_t* fix_u; const int32_t* fix_i; const int32_t* fix_j;   // yue_bpr_adam_apply: the caller's triplets (K = 1)
    uint64_t seed; uint32_t epoch;                 // epoch = the step's index
    float reg, lr_t;
    uint32_t tag;                                  // stamp of this step's touched rows
    // per-step scratch
    int32_t* row_u; int32_t* row_i; int32_t* row_e;   // [B]
    int32_t* trip_j; float* trip_c; float* trip_loss; // [B K]
    float* ucopy; float* ugrad;                    // [B, ld]
    float* row_c; double* row_loss;                // [B]
    int32_t* slot_row; int32_t* slot_pos;          // [2B + B K]: graph row (users first), arrival order in its bucket
    int32_t* list; int32_t* sorted;                // [2B + B K]: the buckets, in arrival order / in slot order
    int32_t* cnt;                                  // [m + n] zero between steps
    int32_t* row_base; int32_t* row_size; uint32_t* stamp;   // [m + n]
    unsigned* bump;                                // bucket allocator
    double* loss_out;                              // this step's loss
};

__device__ __forceinline__ int64_t bpr_adam_slots(const BprAdamParams& p) { return 2 * (int64_t)p.B + (int64_t)p.B * p.K; }

// the event of batch row b: attempt 0 of slot 4095, scaled to [0, T)
__device__ __forceinline__ int64_t bpr_adam_event(uint64_t seed, uint32_t epoch, int b, int64_t T) {
    uint32_t w[4];
    philox4x32_10((uint32_t)b, 0u, epoch, kBprAdamPosSlot << 20, (uint32_t)seed, (uint32_t)(seed >> 32), w);
    return (int64_t)(((uint64_t)w[0] * (uint64_t)T) >> 32);
}

// the triplet (u, i, j) of slot t = b K + k; e = the event (or -1 for the caller's triplets)
__device__ __forceinline__ void bpr_adam_draw(const BprAdamParams& p, int64_t t, int32_t& u, int32_t& i, int32_t& j, int64_t& e) {
    if (p.fix_u) { u = __ldg(p.fix_u + t); i = __ldg(p.fix_i + t); j = __ldg(p.fix_j + t); e = -1; return; }
    const int b = (int)(t / p.K), k = (int)(t - (int64_t)b * p.K);
    e = bpr_adam_event(p.seed, p.epoch, b, p.T);
    u = __ldg(p.ev_user + e);
    i = __ldg(p.ev_items + e);
    if (i < 0) i = __ldg(p.hot_items + (-i - 1));
    const int64_t rb = __ldg(p.uq_indptr + u);
    j = sample_negative(p.seed, p.epoch, (uint64_t)b, (uint32_t)k, (uint32_t)p.n, p.uq_items + rb, (int)(__ldg(p.uq_indptr + u + 1) - rb));
}

// check hook: the batch's events and negatives
__global__ void bpr_adam_sample_kernel(const BprAdamParams p, int32_t* ev_out, int32_t* neg_out) {
    const int64_t N = (int64_t)p.B * p.K;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < N; t += (int64_t)gridDim.x * blockDim.x) {
        int32_t u, i, j; int64_t e;
        bpr_adam_draw(p, t, u, i, j, e);
        neg_out[t] = j;
        if (t % p.K == 0) ev_out[t / p.K] = (int32_t)e;
    }
}

__device__ __forceinline__ void bpr_adam_count(const BprAdamParams& p, int64_t slot, int32_t row) {
    p.slot_row[slot] = row;
    p.slot_pos[slot] = atomicAdd(p.cnt + row, 1);
}

// phase 1: a group of G lanes per triplet
template <int G, int NC>
__global__ void __launch_bounds__(kBprAdamThreads) bpr_adam_triplet_kernel(const BprAdamParams p) {
    const int gl = threadIdx.x % G;
    const unsigned mask = gcn_group_mask<G>();
    const int64_t N = (int64_t)p.B * p.K, tot = (int64_t)gridDim.x * (kBprAdamThreads / G);
    if (blockIdx.x == 0 && threadIdx.x == 0) *p.bump = 0u;
    for (int64_t t = blockIdx.x * (int64_t)(kBprAdamThreads / G) + threadIdx.x / G; t < N; t += tot) {
        int32_t u, i, j; int64_t e;
        bpr_adam_draw(p, t, u, i, j, e);
        GcnVec<G, NC> pu, qi, qj;
        pu.load(p.P + (int64_t)u * p.ld, p.ld, gl);
        qi.load(p.Q + (int64_t)i * p.ld, p.ld, gl);
        qj.load(p.Q + (int64_t)j * p.ld, p.ld, gl);
        const float x = gcn_group_sum<G>(pu.dot_part(qi) - pu.dot_part(qj), mask);
        const float n2 = gcn_group_sum<G>(pu.dot_part(pu) + qi.dot_part(qi) + qj.dot_part(qj), mask);
        if (gl == 0) {
            const float c = 1.f / (1.f + expf(x));                                   // 1 - sigmoid(x)
            const float sp = x > 0.f ? log1pf(expf(-x)) : -x + log1pf(expf(x));      // softplus(-x)
            p.trip_c[t] = c;
            p.trip_loss[t] = sp + 0.5f * p.reg * n2;
            p.trip_j[t] = j;
            const int b = (int)(t / p.K);
            bpr_adam_count(p, 2 * (int64_t)p.B + t, (int32_t)(p.m + j));
            if (t == (int64_t)b * p.K) {
                p.row_u[b] = u; p.row_i[b] = i; p.row_e[b] = (int32_t)e;
                bpr_adam_count(p, b, u);
                bpr_adam_count(p, (int64_t)p.B + b, (int32_t)(p.m + i));
            }
        }
    }
}

// phase 2: a group per batch row -- the user's gradient over its K triplets in k order, C_b, the row's loss, a copy of U_u
template <int G, int NC>
__global__ void __launch_bounds__(kBprAdamThreads) bpr_adam_row_kernel(const BprAdamParams p) {
    const int gl = threadIdx.x % G;
    const int64_t tot = (int64_t)gridDim.x * (kBprAdamThreads / G);
    for (int64_t b = blockIdx.x * (int64_t)(kBprAdamThreads / G) + threadIdx.x / G; b < p.B; b += tot) {
        const int32_t u = p.row_u[b], i = p.row_i[b];
        GcnVec<G, NC> pu, qi, acc;
        pu.load(p.P + (int64_t)u * p.ld, p.ld, gl);
        qi.load(p.Q + (int64_t)i * p.ld, p.ld, gl);
        acc.zero();
        float C = 0.f;
        double ls = 0.0;
        const int64_t t0 = b * p.K;
#pragma unroll 4
        for (int k = 0; k < p.K; ++k) {
            const float c = __ldcg(p.trip_c + t0 + k);
            GcnVec<G, NC> qj; qj.load(p.Q + (int64_t)__ldcg(p.trip_j + t0 + k) * p.ld, p.ld, gl);
            acc.axpy(c, qj);
            C += c;
            ls += (double)__ldcg(p.trip_loss + t0 + k);
        }
        acc.axpy(-C, qi);
        acc.axpy((float)p.K * p.reg, pu);
        acc.store(p.ugrad + b * p.ld, p.ld, gl);
        pu.store(p.ucopy + b * p.ld, p.ld, gl);
        if (gl == 0) { p.row_c[b] = C; p.row_loss[b] = ls; }
    }
}

// phase 3: the slot that arrived first at its row gives the row a bucket (and resets the row's counter); block 0 also sums
// the step's loss over the rows in row order
__global__ void bpr_adam_alloc_kernel(const BprAdamParams p) {
    const int64_t S = bpr_adam_slots(p);
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < S; s += (int64_t)gridDim.x * blockDim.x) {
        if (p.slot_pos[s] != 0) continue;
        const int32_t r = p.slot_row[s];
        const int32_t c = p.cnt[r];
        p.cnt[r] = 0;
        p.row_base[r] = (int32_t)atomicAdd(p.bump, (unsigned)c);
        p.row_size[r] = c;
        p.stamp[r] = p.tag;
    }
    if (blockIdx.x == 0 && threadIdx.x < 32) {
        double a = 0.0;
        for (int b = threadIdx.x; b < p.B; b += 32) a += p.row_loss[b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (threadIdx.x == 0) *p.loss_out = a;
    }
}

// phase 4: every slot into its row's bucket, in arrival order
__global__ void bpr_adam_scatter_kernel(const BprAdamParams p) {
    const int64_t S = bpr_adam_slots(p);
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < S; s += (int64_t)gridDim.x * blockDim.x)
        p.list[p.row_base[p.slot_row[s]] + p.slot_pos[s]] = (int32_t)s;
}

// phase 5: every bucket in slot order (a slot's place = the number of smaller slots in its bucket)
__global__ void bpr_adam_rank_kernel(const BprAdamParams p) {
    const int64_t S = bpr_adam_slots(p);
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < S; s += (int64_t)gridDim.x * blockDim.x) {
        const int32_t r = p.slot_row[s];
        const int32_t base = p.row_base[r], size = p.row_size[r];
        int rank = 0;
        for (int x = 0; x < size; ++x) rank += p.list[base + x] < (int32_t)s;
        p.sorted[base + rank] = (int32_t)s;
    }
}

// phase 6: Adam on every float4 of U and V; a touched row adds its bucket's contributions up in slot order
__global__ void __launch_bounds__(kBprAdamThreads) bpr_adam_update_kernel(const BprAdamParams p) {
    const int per = p.ld / 4;
    const int64_t M = p.m + p.n, total = M * per;
    const float kreg = (float)p.K * p.reg;
    const int B = p.B;
    for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = x / per;
        const int q = (int)(x - r * per);
        float4* var = reinterpret_cast<float4*>((r < p.m ? p.P + r * p.ld : p.Q + (r - p.m) * p.ld) + 4 * q);
        float4* mp = reinterpret_cast<float4*>(p.am + r * p.ld + 4 * q);
        float4* vp = reinterpret_cast<float4*>(p.av + r * p.ld + 4 * q);
        float4 w = __ldcs(var), mo = __ldcs(mp), ve = __ldcs(vp);
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (__ldg(p.stamp + r) == p.tag) {
            const int32_t base = p.row_base[r], size = p.row_size[r];
            for (int z = 0; z < size; ++z) {
                const int32_t s = p.sorted[base + z];
                if (s < B) {                                                       // the user of row s
                    const float4 a = reinterpret_cast<const float4*>(p.ugrad + (int64_t)s * p.ld)[q];
                    g.x += a.x; g.y += a.y; g.z += a.z; g.w += a.w;
                    continue;
                }
                float coef, rg;
                int64_t b;
                if (s < 2 * B) { b = s - B; coef = -p.row_c[b]; rg = kreg; }        // the positive of row b, K times
                else { const int64_t t = s - 2 * (int64_t)B; b = t / p.K; coef = p.trip_c[t]; rg = p.reg; }
                const float4 a = reinterpret_cast<const float4*>(p.ucopy + b * p.ld)[q];
                g.x += fmaf(coef, a.x, rg * w.x); g.y += fmaf(coef, a.y, rg * w.y);
                g.z += fmaf(coef, a.z, rg * w.z); g.w += fmaf(coef, a.w, rg * w.w);
            }
        }
        float* gg = &g.x; float* mm = &mo.x; float* vv = &ve.x; float* xx = &w.x;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            mm[c] = 0.9f * mm[c] + 0.1f * gg[c];
            vv[c] = 0.999f * vv[c] + 0.001f * gg[c] * gg[c];
            xx[c] -= p.lr_t * mm[c] / (sqrtf(vv[c]) + 1e-8f);
        }
        __stcs(var, w); __stcs(mp, mo); __stcs(vp, ve);
    }
}

}  // namespace yue
