// Training-step kernels: fused BPR forward+backward, EmbLoss, dense Adam+L2 sweep, row gather / scatter-add.
// See include/whisprrec_b200.h for the reference lines each entry point replaces.
#include <cmath>
#include <cstring>
#include <type_traits>

#include "common.cuh"

namespace wr {

// ------------------------------------------------------------------------------------------------------
// BPR forward + backward.  One group of LPR lanes per interaction; the three rows stay in registers
// between the dot products and the gradient reductions, so each row is read exactly once.
// ------------------------------------------------------------------------------------------------------
template <class TABS>
struct BprParamsT {
    TABS tabs;
    const int64_t *user, *pos, *neg;
    int64_t B, n_users, n_items;
    float gamma, coef;  // coef = grad_scale / (rows of the whole batch)
    float loss_div;     // rows of the whole batch (= B on one GPU)
    float *loss_out;
    int accumulate_loss;
    WrWorkspace *ws;
};
using BprParams = BprParamsT<LocalTabs>;

// Deterministic epilogue shared by the loss kernels: per-block partials, summed in block order by the last block.
__device__ __forceinline__ void finish_loss(float local, float *red, bool *flag, WrWorkspace *ws, int slot,
                                            float B, float *loss_out, int accumulate) {
    const float bsum = block_sum(local, red);
    if (threadIdx.x == 0) ws->partial[slot * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = bsum;
    if (last_block_arrives(&ws->ticket[slot], flag)) {
        if (threadIdx.x < 32) {
            float t = 0.f;
            for (int i = threadIdx.x; i < (int)gridDim.x; i += 32)
                t += __ldcg(&ws->partial[slot * WR_MAX_PARTIAL_BLOCKS + i]);
            t = warp_sum(t);
            if (threadIdx.x == 0) {
                const float mean = t / B;
                loss_out[0] = accumulate ? loss_out[0] + mean : mean;
            }
        }
    }
}

template <int LPR, int VPL, class TABS>
__global__ void __launch_bounds__(256) bpr_fwd_bwd_kernel(BprParamsT<TABS> p) {
    using RG = RowGroup<LPR, VPL>;
    constexpr int D = RG::D;
    __shared__ float red[8];
    __shared__ bool flag;
    const int lane = threadIdx.x & 31, sub = lane % LPR, grp = lane / LPR;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    float local = 0.f;
    for (int64_t base = warp * RG::GROUPS; base < p.B; base += nwarps * RG::GROUPS) {
        const int64_t b = base + grp;
        const bool valid = b < p.B;
        int64_t u = 0, i = 0, j = 0;
        if (valid) {
            u = p.user[b];
            i = p.pos[b];
            j = p.neg[b];
        }
        const bool ok = valid && (uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
                        (uint64_t)j < (uint64_t)p.n_items;
        if (valid && !ok && sub == 0) atomicOr(&p.ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
        float4 ue[VPL], pe[VPL], ne[VPL];
        if (ok) {
            RG::load(p.tabs.row(b, 0, u, D), sub, ue);
            RG::load(p.tabs.row(b, 1, i, D), sub, pe);
            RG::load(p.tabs.row(b, 2, j, D), sub, ne);
        } else {
            RG::zero(ue);
            RG::zero(pe);
            RG::zero(ne);
        }
        float sp = 0.f, sn = 0.f;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            sp += dot4(ue[v], pe[v]);
            sn += dot4(ue[v], ne[v]);
        }
        sp = group_sum<LPR>(sp);
        sn = group_sum<LPR>(sn);
        if (ok) {
            float l, c;
            bpr_pointwise(sp, sn, p.gamma, p.coef, l, c);
            if (sub == 0) local += l;
#pragma unroll
            for (int v = 0; v < VPL; ++v) {
                const int off = 4 * (sub + v * LPR);
                p.tabs.add_user(u, D, off, scale4(sub4(pe[v], ne[v]), c), b, 0);
                p.tabs.add_item(i, D, off, scale4(ue[v], c), b, 1);
                p.tabs.add_item(j, D, off, scale4(ue[v], -c), b, 2);
            }
        }
    }
    finish_loss(local, red, &flag, p.ws, 0, p.loss_div, p.loss_out, p.accumulate_loss);
}

// Any D % 4 == 0: a warp per interaction, rows re-read for the gradient (they are L1 hits).
template <class TABS>
__global__ void __launch_bounds__(256) bpr_fwd_bwd_generic_kernel(BprParamsT<TABS> p, int D) {
    __shared__ float red[8];
    __shared__ bool flag;
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int D4 = D >> 2;
    float local = 0.f;
    for (int64_t b = warp; b < p.B; b += nwarps) {
        const int64_t u = p.user[b], i = p.pos[b], j = p.neg[b];
        const bool ok = (uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
                        (uint64_t)j < (uint64_t)p.n_items;
        if (!ok) {
            if (lane == 0) atomicOr(&p.ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
            continue;
        }
        const float *ur = p.tabs.urow(u, D), *pr = p.tabs.irow(i, D), *nr = p.tabs.irow(j, D);
        float *gu = p.tabs.gurow(u, D), *gp = p.tabs.girow(i, D), *gn = p.tabs.girow(j, D);
        float sp = 0.f, sn = 0.f;
        for (int v = lane; v < D4; v += 32) {
            const float4 a = ldg4(ur + 4 * v);
            sp += dot4(a, ldg4(pr + 4 * v));
            sn += dot4(a, ldg4(nr + 4 * v));
        }
        sp = warp_sum(sp);
        sn = warp_sum(sn);
        float l, c;
        bpr_pointwise(sp, sn, p.gamma, p.coef, l, c);
        if (lane == 0) local += l;
        for (int v = lane; v < D4; v += 32) {
            const float4 a = ldg4(ur + 4 * v), x = ldg4(pr + 4 * v), y = ldg4(nr + 4 * v);
            red_add_v4(gu + 4 * v, scale4(sub4(x, y), c));
            red_add_v4(gp + 4 * v, scale4(a, c));
            red_add_v4(gn + 4 * v, scale4(a, -c));
        }
    }
    finish_loss(local, red, &flag, p.ws, 0, p.loss_div, p.loss_out, p.accumulate_loss);
}

// ------------------------------------------------------------------------------------------------------
// EmbLoss: phase 1 sums squares of the gathered ego rows (per occurrence), phase 2 scatters row/||.||.
// ------------------------------------------------------------------------------------------------------
template <class TABS>
struct EmbParamsT {
    TABS tabs;
    const int64_t *user, *pos, *neg;
    int64_t B, n_users, n_items;
    float reg_weight;
    float inv_rows;          // 1 / rows of the whole batch
    float *loss_out;         // nullable
    float *sumsq_out;        // sharded: this rank's three sums of squares go here instead of ws->norms
    const float *sumsq_in;   // sharded: the three GLOBAL sums of squares
    WrWorkspace *ws;
};
using EmbParams = EmbParamsT<LocalTabs>;

template <class TABS>
__global__ void __launch_bounds__(256) embloss_sumsq_kernel(EmbParamsT<TABS> p, int D) {
    __shared__ float red[8];
    __shared__ bool flag;
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int D4 = D >> 2;
    float su = 0.f, sp = 0.f, sn = 0.f;
    // lanes cover (interaction, float4) pairs so that D=64 rows keep all 32 lanes busy
    const int64_t total = p.B * D4;
    for (int64_t t = warp * 32 + lane; t < total; t += nwarps * 32) {
        const int64_t b = t / D4;
        const int v = (int)(t - b * D4);
        const int64_t u = p.user[b], i = p.pos[b], j = p.neg[b];
        if ((uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
            (uint64_t)j < (uint64_t)p.n_items) {
            const float4 a = ldg4(p.tabs.urow(u, D) + 4 * v), x = ldg4(p.tabs.irow(i, D) + 4 * v),
                         y = ldg4(p.tabs.irow(j, D) + 4 * v);
            su += dot4(a, a);
            sp += dot4(x, x);
            sn += dot4(y, y);
        }
    }
    const float bu = block_sum(su, red), bp = block_sum(sp, red), bn = block_sum(sn, red);
    if (threadIdx.x == 0) {
        p.ws->partial[0 * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = bu;
        p.ws->partial[1 * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = bp;
        p.ws->partial[2 * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = bn;
    }
    if (last_block_arrives(&p.ws->ticket[1], &flag)) {
        if (threadIdx.x < 32) {
            float t[3] = {0.f, 0.f, 0.f};
            for (int i = threadIdx.x; i < (int)gridDim.x; i += 32)
#pragma unroll
                for (int q = 0; q < 3; ++q) t[q] += __ldcg(&p.ws->partial[q * WR_MAX_PARTIAL_BLOCKS + i]);
#pragma unroll
            for (int q = 0; q < 3; ++q) t[q] = warp_sum(t[q]);
            if (threadIdx.x == 0) {
                if (p.sumsq_out) {      // the norms are batch-global: the ranks' sums meet before the square root
                    p.sumsq_out[0] = t[0];
                    p.sumsq_out[1] = t[1];
                    p.sumsq_out[2] = t[2];
                } else {
                    t[0] = sqrtf(t[0]);
                    t[1] = sqrtf(t[1]);
                    t[2] = sqrtf(t[2]);
                    p.ws->norms[0] = t[0];
                    p.ws->norms[1] = t[1];
                    p.ws->norms[2] = t[2];
                    // utils/loss.py:94-98: (sum of the three norms) / B, scaled by reg_weight at LightGCN.py:175
                    p.loss_out[0] += p.reg_weight * ((t[0] + t[1] + t[2]) * p.inv_rows);
                }
            }
        }
    }
}

template <class TABS>
__global__ void __launch_bounds__(256) embloss_scatter_kernel(EmbParamsT<TABS> p, int D) {
    const int D4 = D >> 2;
    const float k = p.reg_weight * p.inv_rows;
    float nu, np_, nn;
    if (p.sumsq_in) {
        nu = sqrtf(p.sumsq_in[0]);
        np_ = sqrtf(p.sumsq_in[1]);
        nn = sqrtf(p.sumsq_in[2]);
        if (p.loss_out && blockIdx.x == 0 && threadIdx.x == 0) p.loss_out[0] += p.reg_weight * ((nu + np_ + nn) * p.inv_rows);
    } else {
        nu = p.ws->norms[0];
        np_ = p.ws->norms[1];
        nn = p.ws->norms[2];
    }
    const float ku = nu > 0.f ? k / nu : 0.f, kp = np_ > 0.f ? k / np_ : 0.f, kn = nn > 0.f ? k / nn : 0.f;
    const int64_t total = p.B * D4;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = t / D4;
        const int v = (int)(t - b * D4);
        const int64_t u = p.user[b], i = p.pos[b], j = p.neg[b];
        if ((uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
            (uint64_t)j < (uint64_t)p.n_items) {
            red_add_v4(p.tabs.gurow(u, D) + 4 * v, scale4(ldg4(p.tabs.urow(u, D) + 4 * v), ku));
            red_add_v4(p.tabs.girow(i, D) + 4 * v, scale4(ldg4(p.tabs.irow(i, D) + 4 * v), kp));
            red_add_v4(p.tabs.girow(j, D) + 4 * v, scale4(ldg4(p.tabs.irow(j, D) + 4 * v), kn));
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// Dense Adam with coupled L2 and fused zero_grad: one streaming pass, 32 B of traffic per parameter.
// ------------------------------------------------------------------------------------------------------
template <int UNROLL>
__global__ void __launch_bounds__(256) adam_sweep_kernel(float4 *__restrict__ P, float4 *__restrict__ M,
                                                          float4 *__restrict__ V, float4 *__restrict__ G,
                                                          int64_t n4, AdamScalars s, const float *dev_scalars) {
    if (dev_scalars) {
        s.step_size = __ldg(dev_scalars);
        s.bc2_sqrt = __ldg(dev_scalars + 1);
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const float4 z = f4_zero();
    for (; i + (UNROLL - 1) * stride < n4; i += UNROLL * stride) {
        float4 p[UNROLL], m[UNROLL], v[UNROLL], g[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            p[u] = P[i + u * stride];
            m[u] = M[i + u * stride];
            v[u] = V[i + u * stride];
            g[u] = G[i + u * stride];
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            adam_elem(p[u].x, m[u].x, v[u].x, g[u].x, s);
            adam_elem(p[u].y, m[u].y, v[u].y, g[u].y, s);
            adam_elem(p[u].z, m[u].z, v[u].z, g[u].z, s);
            adam_elem(p[u].w, m[u].w, v[u].w, g[u].w, s);
            P[i + u * stride] = p[u];
            M[i + u * stride] = m[u];
            V[i + u * stride] = v[u];
            G[i + u * stride] = z;
        }
    }
    for (; i < n4; i += stride) {
        float4 p = P[i], m = M[i], v = V[i], g = G[i];
        adam_elem(p.x, m.x, v.x, g.x, s);
        adam_elem(p.y, m.y, v.y, g.y, s);
        adam_elem(p.z, m.z, v.z, g.z, s);
        adam_elem(p.w, m.w, v.w, g.w, s);
        P[i] = p;
        M[i] = m;
        V[i] = v;
        G[i] = z;
    }
}

__global__ void adam_tail_kernel(float *P, float *M, float *V, float *G, int64_t from, int64_t n, AdamScalars s,
                                 const float *dev_scalars) {
    if (dev_scalars) {
        s.step_size = dev_scalars[0];
        s.bc2_sqrt = dev_scalars[1];
    }
    const int64_t i = from + threadIdx.x;
    if (i < n) {
        adam_elem(P[i], M[i], V[i], G[i], s);
        G[i] = 0.f;
    }
}

// The same sweep for a gradient that is zero outside a few rows (BPRMF: the 3 B rows of the batch): bit r of `touched`
// says row r of G holds something.  Rows whose bit is clear are updated with g = 0 and their G row is neither read nor
// rewritten: 24 B of traffic per parameter instead of 32.  `shift` = log2(D/4) when D/4 is a power of two, else -1.
template <int UNROLL>
__global__ void __launch_bounds__(256) adam_sweep_marked_kernel(float4 *__restrict__ P, float4 *__restrict__ M,
                                                                 float4 *__restrict__ V, float4 *__restrict__ G,
                                                                 int64_t n4, int D4, int shift,
                                                                 const uint32_t *__restrict__ touched, AdamScalars s,
                                                                 const float *dev_scalars) {
    if (dev_scalars) {
        s.step_size = __ldg(dev_scalars);
        s.bc2_sqrt = __ldg(dev_scalars + 1);
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const float4 z = f4_zero();
    for (; i < n4; i += UNROLL * stride) {
        float4 p[UNROLL], m[UNROLL], v[UNROLL], g[UNROLL];
        bool hit[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int64_t e = i + u * stride;
            hit[u] = false;
            if (e < n4) {
                const int64_t row = shift >= 0 ? (e >> shift) : (e / D4);
                hit[u] = (__ldg(touched + (row >> 5)) >> (row & 31)) & 1u;
                p[u] = P[e];
                m[u] = M[e];
                v[u] = V[e];
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) g[u] = hit[u] ? G[i + u * stride] : z;
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int64_t e = i + u * stride;
            if (e < n4) {
                adam_elem(p[u].x, m[u].x, v[u].x, g[u].x, s);
                adam_elem(p[u].y, m[u].y, v[u].y, g[u].y, s);
                adam_elem(p[u].z, m[u].z, v[u].z, g[u].z, s);
                adam_elem(p[u].w, m[u].w, v[u].w, g[u].w, s);
                P[e] = p[u];
                M[e] = m[u];
                V[e] = v[u];
                if (hit[u]) G[e] = z;
            }
        }
    }
}

// Bits of the rows a batch touches, in the concatenated [users; items] numbering (out-of-range ids are the gradient
// kernel's to report).
__global__ void __launch_bounds__(256) mark_rows_kernel(const int64_t *user, const int64_t *pos, const int64_t *neg,
                                                         int64_t B, int64_t n_users, int64_t n_items, uint32_t *touched) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int64_t u = user[b], i = pos[b], j = neg[b];
    if ((uint64_t)u >= (uint64_t)n_users || (uint64_t)i >= (uint64_t)n_items || (uint64_t)j >= (uint64_t)n_items) return;
    const int64_t r1 = n_users + i, r2 = n_users + j;
    atomicOr(touched + (u >> 5), 1u << (u & 31));
    atomicOr(touched + (r1 >> 5), 1u << (r1 & 31));
    atomicOr(touched + (r2 >> 5), 1u << (r2 & 31));
}

// ------------------------------------------------------------------------------------------------------
// Row movement for row-sharded tables.
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_rows_kernel(const float *__restrict__ T, const int64_t *idx,
                                                           int64_t B, int D, int64_t n_rows, float *out,
                                                           WrWorkspace *ws) {
    const int D4 = D >> 2;
    const int64_t total = B * D4;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = t / D4;
        const int v = (int)(t - b * D4);
        const int64_t r = idx[b];
        float4 x = f4_zero();
        if ((uint64_t)r < (uint64_t)n_rows)
            x = ldg4(T + r * D + 4 * v);
        else if (v == 0)
            atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
        reinterpret_cast<float4 *>(out)[t] = x;
    }
}

__global__ void __launch_bounds__(256) scatter_add_rows_kernel(float *G, const int64_t *idx, int64_t B, int D,
                                                                int64_t n_rows, const float *__restrict__ rows,
                                                                WrWorkspace *ws) {
    const int D4 = D >> 2;
    const int64_t total = B * D4;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = t / D4;
        const int v = (int)(t - b * D4);
        const int64_t r = idx[b];
        if ((uint64_t)r < (uint64_t)n_rows)
            red_add_v4(G + r * D + 4 * v, ldg4(rows + t * 4));
        else if (v == 0)
            atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
    }
}

// ------------------------------------------------------------------------------------------------------
// One launch for a whole BPRMF step (BaseRunner.py:196-199) when the tables are cache-sized and the step is
// latency-bound rather than bandwidth-bound: every warp first issues its ids, then the CTA pulls its spans of
// P / M / V / G towards L2 (they do not depend on the batch), the grid does the BPR forward+backward (ids -> rows ->
// REDs into G) while those streams are in flight, meets at a grid barrier (cooperative launch: all CTAs are
// resident), and finishes with the Adam+L2 update of its spans, which come back as L2 hits.
// ------------------------------------------------------------------------------------------------------
// Cross-GPU synchronisation state of the single-launch step on row-sharded tables (world > 1).
struct StepSync {
    uint32_t *flags[WR_MAX_WORLD];  // rank g's [2][WR_MAX_WORLD] words: [0][r] = r's gradients have landed (epoch e),
                                    //                                  [1][r] = r's Adam of step e is complete
    float *slots[WR_MAX_WORLD];     // rank g's [2 (epoch parity)][WR_MAX_WORLD] loss shares
    int world, rank;
    uint32_t epoch;                 // the step number: 1, 2, 3, ... (the same on every rank)
};

// wr_debug_step_trace: [CTA][8] %globaltimer stamps of thread 0 of every CTA, written by the TRACE instantiation only
// (the production instantiation never names it).  Slots: 0 entry, 1 ids landed, 2 rows landed, 3 REDs issued,
// 4 arrived (fence + arrival done), 5 barrier passed, 6 Adam operands landed, 7 exit.  Slots 1 / 2 / 6 are thread 0's
// last batch group and last Adam iteration.
__device__ uint64_t *g_step_trace;

__device__ __forceinline__ void wait_for(int64_t x) { asm volatile("" ::"l"(x)); }
__device__ __forceinline__ void wait_for(float4 x) { asm volatile("" ::"f"(x.x), "f"(x.y), "f"(x.z), "f"(x.w)); }

// The stamp waits for `deps` (registers of loads that must have landed) before it reads the clock.
template <bool TRACE, class... T>
__device__ __forceinline__ void step_stamp(int slot, T... deps) {
    if constexpr (TRACE) {
        if (threadIdx.x == 0) {
            (wait_for(deps), ...);
            g_step_trace[8 * blockIdx.x + slot] = global_timer_ns();
        }
    }
}

// Wait until CTA `line`'s arrival word has reached `value` (wrap-safe); gives up after WR_PEER_TIMEOUT_NS so that a CTA
// that never arrives cannot hang the GPU.
__device__ __forceinline__ void wait_arrival(const uint32_t *line, uint32_t value, WrWorkspace *ws) {
    uint64_t t0 = 0;
    for (uint32_t spins = 1; (int32_t)(ld_acquire_u32(line) - value) < 0; ++spins) {
        if ((spins & 1023u) == 0) {
            const uint64_t now = global_timer_ns();
            if (t0 == 0) t0 = now;
            if (now - t0 > WR_PEER_TIMEOUT_NS) {
                atomicOr(&ws->status, WR_STATUS_PEER_TIMEOUT);
                break;
            }
        }
    }
}

// One CTA per SM (launch_step_fused sizes blockDim so that every thread's Adam share is whole).
template <int LPR, int VPL, class TABS, bool TRACE = false>
__global__ void __launch_bounds__(1024, 1) bprmf_step_kernel(BprParamsT<TABS> p, float4 *P, float4 *M, float4 *V, float4 *G,
                                                             int64_t n4, AdamScalars s, const float *dev_scalars,
                                                             StepSync sy) {
    using RG = RowGroup<LPR, VPL>;
    constexpr int D = RG::D;
    __shared__ float red[32];
    step_stamp<TRACE>(0);
    // The grid barrier's generation: every CTA reads it before it arrives, CTA 0 advances it once it has passed, so
    // arrival lines need no reset and a line left by an earlier launch (of any grid size) is simply older.
    const uint32_t arrived = ld_relaxed_gpu_u32(&p.ws->st_gen) + 1u;
    if (dev_scalars) {
        s.step_size = __ldg(dev_scalars);
        s.bc2_sqrt = __ldg(dev_scalars + 1);
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // The first batch group's ids go out before the table streams below: behind 10 MB of them in the DRAM queues they
    // land microseconds later, and every gather waits for them.
    const int lane = threadIdx.x & 31, sub = lane % LPR, grp = lane / LPR;
    const int64_t warp = (int64_t)(threadIdx.x >> 5) * gridDim.x + blockIdx.x;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t first = warp * RG::GROUPS;
    int64_t u = 0, i = 0, j = 0;
    if (first + grp < p.B) {
        u = p.user[first + grp];
        i = p.pos[first + grp];
        j = p.neg[first + grp];
    }
    // ---- phase 0: pull this CTA's spans of P / M / V / G towards L2 (one bulk prefetch per span) ----
    if (threadIdx.x < 4) {      // G too: the gradient REDs then meet lines that are already on their way
        const float4 *arr = threadIdx.x == 0 ? P : (threadIdx.x == 1 ? M : (threadIdx.x == 2 ? V : G));
        for (int64_t c = (int64_t)blockIdx.x * blockDim.x; c < n4; c += stride) {
            const uint32_t bytes = (uint32_t)min((int64_t)blockDim.x, n4 - c) * 16u;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(arr + c), "r"(bytes) : "memory");
        }
    }
    if (sy.world > 1) {
        // remote rows may be gathered only once their owners have finished the previous step's Adam
        if (threadIdx.x < sy.world) {
            const uint64_t t0 = global_timer_ns();
            while ((int32_t)(ld_acquire_sys(sy.flags[sy.rank] + WR_MAX_WORLD + threadIdx.x) - (sy.epoch - 1u)) < 0) {
                if (global_timer_ns() - t0 > WR_PEER_TIMEOUT_NS) {
                    atomicOr(&p.ws->status, WR_STATUS_PEER_TIMEOUT);
                    break;
                }
            }
        }
        __syncthreads();
    }
    // ---- phase 1: BPR forward + backward; consecutive interaction groups go to different CTAs ----
    float local = 0.f;
    for (int64_t base = first; base < p.B; base += nwarps * RG::GROUPS) {
        const int64_t b = base + grp;
        const bool valid = b < p.B;
        if (base != first) {
            u = i = j = 0;
            if (valid) {
                u = p.user[b];
                i = p.pos[b];
                j = p.neg[b];
            }
        }
        const bool ok = valid && (uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
                        (uint64_t)j < (uint64_t)p.n_items;
        step_stamp<TRACE>(1, j);                   // (the last of the three id loads)
        if (valid && !ok && sub == 0) atomicOr(&p.ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
        float4 ue[VPL], pe[VPL], ne[VPL];
        if (ok) {     // P is rewritten by phase 2 (and by the peers' Adam phases): coherent loads, not ld.global.nc
            RG::load_cg(p.tabs.urow(u, D), sub, ue);
            RG::load_cg(p.tabs.irow(i, D), sub, pe);
            RG::load_cg(p.tabs.irow(j, D), sub, ne);
        } else {
            RG::zero(ue);
            RG::zero(pe);
            RG::zero(ne);
        }
        step_stamp<TRACE>(2, ne[VPL - 1]);         // (the last of the row loads)
        float sp = 0.f, sn = 0.f;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            sp += dot4(ue[v], pe[v]);
            sn += dot4(ue[v], ne[v]);
        }
        sp = group_sum<LPR>(sp);
        sn = group_sum<LPR>(sn);
        if (ok) {
            float l, c;
            bpr_pointwise(sp, sn, p.gamma, p.coef, l, c);
            if (sub == 0) local += l;
            float *gu = p.tabs.gurow(u, D), *gp = p.tabs.girow(i, D), *gn = p.tabs.girow(j, D);
#pragma unroll
            for (int v = 0; v < VPL; ++v) {
                const int off = 4 * (sub + v * LPR);
                red_add_v4(gu + off, scale4(sub4(pe[v], ne[v]), c));
                red_add_v4(gp + off, scale4(ue[v], c));
                red_add_v4(gn + off, scale4(ue[v], -c));
            }
        }
    }
    // block_sum's last __syncthreads follows every REDs of the CTA: thread 0's release below speaks for all of them
    const float bsum = block_sum(local, red);
    step_stamp<TRACE>(3);
    // ---- grid barrier: CTA c release-stores the generation + 1 into its own 128-byte line (after its REDs, and its
    //      loss partial), thread t waits for lines t, t + blockDim, ...: no counter, no atomics.  (Small tables run
    //      more CTAs than threads: (500 + 700) x 64 is 100 CTAs of 96.)  Sharded: only CTA 0 waits; once every
    //      local CTA has arrived (all of this GPU's REDs, local and remote, are performed) it deposits the loss share
    //      with every peer, publishes this rank's arrival, waits for every peer's, and only then opens the gate
    //      (ticket[5]) for the local CTAs. ----
    if (threadIdx.x == 0) {
        p.ws->partial[blockIdx.x] = bsum;
        if (sy.world > 1) __threadfence_system();
        st_release_gpu(&p.ws->st_flag[32 * blockIdx.x], arrived);
        step_stamp<TRACE>(4);
    }
    if (sy.world == 1 || blockIdx.x == 0) {
        for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) wait_arrival(&p.ws->st_flag[32 * c], arrived, p.ws);
        __syncthreads();
    }
    if (blockIdx.x == 0) {
        float loss_sum = 0.f;
        if (threadIdx.x < 32) {      // this GPU's loss share, summed in CTA order (deterministic)
            if (threadIdx.x == 0) p.ws->st_gen = arrived;      // every CTA read the generation before it arrived
            float t = 0.f;
            for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) t += __ldcg(&p.ws->partial[i]);
            loss_sum = warp_sum(t) / p.loss_div;
        }
        if (sy.world > 1) {
            // Arrival and loss share travel as ONE 8-byte word {epoch, loss bits} per peer (slots[g] read as uint64[world]):
            // no fence between a payload and its flag (a fence.sys behind a remote store is an NVLink round trip).  The
            // word is a release: every local CTA fenced its REDs at system scope before the line this CTA acquired.
            // One slot per sender suffices: a peer writes epoch e + 1 only after it has seen this rank's rows-final flag
            // of epoch e, which is published after the losses of epoch e were read.
            loss_sum = __shfl_sync(0xffffffffu, loss_sum, 0);
            if (threadIdx.x < sy.world) {
                const int g = threadIdx.x;
                __threadfence_system();
                unsigned long long *dst = reinterpret_cast<unsigned long long *>(sy.slots[g]) + sy.rank;
                const unsigned long long word = ((unsigned long long)__float_as_uint(loss_sum) << 32) | sy.epoch;
                asm volatile("st.relaxed.sys.global.b64 [%0], %1;" ::"l"(dst), "l"(word) : "memory");
                const unsigned long long *src = reinterpret_cast<const unsigned long long *>(sy.slots[sy.rank]) + g;
                const uint64_t t0 = global_timer_ns();
                float got = 0.f;
                for (;;) {
                    unsigned long long w;
                    asm volatile("ld.acquire.sys.global.b64 %0, [%1];" : "=l"(w) : "l"(src) : "memory");
                    if ((int32_t)((uint32_t)w - sy.epoch) >= 0) {
                        got = __uint_as_float((uint32_t)(w >> 32));
                        break;
                    }
                    if (global_timer_ns() - t0 > WR_PEER_TIMEOUT_NS) {      // the peer is gone: do not hang the GPU
                        atomicOr(&p.ws->status, WR_STATUS_PEER_TIMEOUT);
                        break;
                    }
                }
                red[threadIdx.x] = got;          // (`red` is free again: block_sum finished before the barrier above)
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                float t = 0.f;
                for (int g = 0; g < sy.world; ++g) t += red[g];      // rank order: the same sum on every rank
                loss_sum = t;
                __threadfence();
                st_release_gpu(&p.ws->ticket[5], sy.epoch);     // the gate: every rank's gradients have landed
            }
        }
        if (threadIdx.x == 0) {
            p.loss_out[0] = p.accumulate_loss ? p.loss_out[0] + loss_sum : loss_sum;
        }
    } else if (sy.world > 1) {
        if (threadIdx.x == 0) {
            uint64_t t0 = 0;
            for (uint32_t spins = 1; ld_acquire_u32(&p.ws->ticket[5]) != sy.epoch; ++spins) {
                if ((spins & 1023u) == 0) {
                    const uint64_t now = global_timer_ns();
                    if (t0 == 0) t0 = now;
                    if (now - t0 > 2 * WR_PEER_TIMEOUT_NS) {
                        atomicOr(&p.ws->status, WR_STATUS_PEER_TIMEOUT);
                        break;
                    }
                }
            }
            __threadfence();
        }
    }
    if (sy.world > 1) __syncthreads();
    step_stamp<TRACE>(5);
    // ---- phase 2: Adam + L2 over every element, gradient re-zeroed; two iterations of loads in flight ----
    // div_nr / sqrt_nr (<= 1 ulp from the IEEE forms): with the IEEE sequences this phase is issue-bound on cache-sized tables
    const float inv_bc2 = 1.0f / s.bc2_sqrt;
    const float4 z = f4_zero();
    for (int64_t i = i0; i < n4; i += 2 * stride) {
        const int64_t i2 = i + stride;
        const bool two = i2 < n4;
        float4 pa = P[i], ma = M[i], va = V[i], ga = __ldcg(G + i);
        float4 pb = z, mb = z, vb = z, gb = z;
        if (two) {
            pb = P[i2];
            mb = M[i2];
            vb = V[i2];
            gb = __ldcg(G + i2);
        }
        step_stamp<TRACE>(6, ga, gb);
        adam_elem_nr(pa.x, ma.x, va.x, ga.x, s, inv_bc2);
        adam_elem_nr(pa.y, ma.y, va.y, ga.y, s, inv_bc2);
        adam_elem_nr(pa.z, ma.z, va.z, ga.z, s, inv_bc2);
        adam_elem_nr(pa.w, ma.w, va.w, ga.w, s, inv_bc2);
        P[i] = pa;
        M[i] = ma;
        V[i] = va;
        G[i] = z;
        if (two) {
            adam_elem_nr(pb.x, mb.x, vb.x, gb.x, s, inv_bc2);
            adam_elem_nr(pb.y, mb.y, vb.y, gb.y, s, inv_bc2);
            adam_elem_nr(pb.z, mb.z, vb.z, gb.z, s, inv_bc2);
            adam_elem_nr(pb.w, mb.w, vb.w, gb.w, s, inv_bc2);
            P[i2] = pb;
            M[i2] = mb;
            V[i2] = vb;
            G[i2] = z;
        }
    }
    // Sharded: the last CTA to finish its Adam tells the peers that this rank's rows of P are final (they may gather
    // them for step e + 1).  One GPU: nothing reads a departure, the next launch starts behind this one in stream order.
    if (sy.world > 1) {
        __syncthreads();                        // the departure below speaks for the whole CTA's stores
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(&p.ws->ticket[4], 1u) == gridDim.x - 1) {
                p.ws->ticket[4] = 0;
                // ONE fence, then relaxed stores that travel side by side (a release store per peer waits for the
                // previous peer's acknowledgement: world - 1 serialised NVLink round trips on the next step's critical path)
                __threadfence_system();
                for (int g = 0; g < sy.world; ++g)
                    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(sy.flags[g] + WR_MAX_WORLD + sy.rank), "r"(sy.epoch)
                                 : "memory");
            }
        }
    }
    step_stamp<TRACE>(7);
}

static inline int grid_for(int64_t work_items, int per_block, int max_blocks) {
    int64_t g = (work_items + per_block - 1) / per_block;
    if (g < 1) g = 1;
    if (g > max_blocks) g = max_blocks;
    return (int)g;
}

template <class TABS>
static int launch_bpr(BprParamsT<TABS> &p, int D, cudaStream_t st) {
#define WR_BPR_CALL(LPR, VPL)                                                              \
    {                                                                                      \
        const int per_block = 8 * (32 / LPR);                                              \
        const int grid = grid_for(p.B, per_block, 8 * kSMs);                               \
        bpr_fwd_bwd_kernel<LPR, VPL, TABS><<<grid, 256, 0, st>>>(p);                       \
    }
    switch (D) {
        case 16: WR_BPR_CALL(4, 1) break;
        case 32: WR_BPR_CALL(8, 1) break;
        case 64: WR_BPR_CALL(16, 1) break;
        case 128: WR_BPR_CALL(32, 1) break;
        case 256: WR_BPR_CALL(32, 2) break;
        default: {
            const int grid = grid_for(p.B, 8, 8 * kSMs);
            bpr_fwd_bwd_generic_kernel<TABS><<<grid, 256, 0, st>>>(p, D);
        }
    }
#undef WR_BPR_CALL
    WR_CHECK_LAUNCH();
    return WR_OK;
}

}  // namespace wr

using namespace wr;

int wr_bprmf_step_impl(float *P, float *M, float *V, float *G, const int64_t *user, const int64_t *pos,
                       const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items, float gamma, float l2,
                       double beta1, double beta2, float eps, float step_size, float bc2_sqrt, const float *dev_scalars,
                       float *loss_out, void *ws, void *stream);

int wr_check_shards(const wr_shards *s) {
    if (s->world < 1 || s->world > WR_MAX_WORLD || s->rank < 0 || s->rank >= s->world) return WR_E_SIZE;
    if (s->n_users <= 0 || s->n_items <= 0 || s->n_users >= INT32_MAX || s->n_items >= INT32_MAX) return WR_E_SIZE;
    if (s->rows_u_local != (s->n_users + s->world - 1) / s->world) return WR_E_SIZE;
    if (s->rows_i_local != (s->n_items + s->world - 1) / s->world) return WR_E_SIZE;
    for (int g = 0; g < s->world; ++g) {
        if (!s->base[g]) return WR_E_NULL;
        if (!wr_aligned16(s->base[g])) return WR_E_ALIGN;
    }
    return WR_OK;
}

extern "C" int wr_bpr_fwd_bwd(const float *U, const float *I, const int64_t *user, const int64_t *pos,
                              const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items, float gamma,
                              float grad_scale, float *gU, float *gI, float *loss_out, int accumulate_loss,
                              void *ws, void *stream) {
    if (!U || !I || !user || !pos || !neg || !gU || !gI || !loss_out || !ws) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(U) || !wr_aligned16(I) || !wr_aligned16(gU) || !wr_aligned16(gI)) return WR_E_ALIGN;
    BprParams p{{U, I, gU, gI}, user, pos, neg, B, n_users, n_items, gamma, grad_scale / (float)B, (float)B,
                loss_out, accumulate_loss, (WrWorkspace *)ws};
    return launch_bpr(p, D, (cudaStream_t)stream);
}

// SGL's BPR term (SGL.py:176-185): sum_b -logsigmoid(s+ - s-), no 1/B; gradient scaled by grad_scale.
extern "C" int wr_bpr_logsig_sum_fwd_bwd(const float *U, const float *I, const int64_t *user, const int64_t *pos,
                                         const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items,
                                         float grad_scale, float *gU, float *gI, float *loss_out, int accumulate_loss,
                                         void *ws, void *stream) {
    if (!U || !I || !user || !pos || !neg || !gU || !gI || !loss_out || !ws) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(U) || !wr_aligned16(I) || !wr_aligned16(gU) || !wr_aligned16(gI)) return WR_E_ALIGN;
    BprParams p{{U, I, gU, gI}, user, pos, neg, B, n_users, n_items, -1.0f /* logsigmoid form */, grad_scale, 1.0f,
                loss_out, accumulate_loss, (WrWorkspace *)ws};
    return launch_bpr(p, D, (cudaStream_t)stream);
}

extern "C" int wr_bpr_fwd_bwd_sharded(const wr_shards *host_T, const wr_shards *host_Gd, const int64_t *user,
                                      const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global, int D,
                                      float gamma, float grad_scale, float *loss_out, void *ws, void *stream) {
    if (!host_T || !host_Gd || !user || !pos || !neg || !loss_out || !ws) return WR_E_NULL;
    int rc = wr_check_shards(host_T);
    if (rc) return rc;
    rc = wr_check_shards(host_Gd);
    if (rc) return rc;
    if (B <= 0 || B_global < B) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    BprParamsT<ShardTabs> p{{*host_T, *host_Gd}, user, pos, neg, B, host_T->n_users, host_T->n_items, gamma,
                            grad_scale / (float)B_global, (float)B_global, loss_out, 0, (WrWorkspace *)ws};
    return launch_bpr(p, D, (cudaStream_t)stream);
}

extern "C" int wr_embloss_fwd_bwd(const float *U0, const float *I0, const int64_t *user, const int64_t *pos,
                                  const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items,
                                  float reg_weight, float *gU0, float *gI0, float *loss_out, void *ws,
                                  void *stream) {
    if (!U0 || !I0 || !user || !pos || !neg || !gU0 || !gI0 || !loss_out || !ws) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(U0) || !wr_aligned16(I0) || !wr_aligned16(gU0) || !wr_aligned16(gI0)) return WR_E_ALIGN;
    EmbParams p{{U0, I0, gU0, gI0}, user, pos, neg, B, n_users, n_items, reg_weight, 1.0f / (float)B, loss_out,
                nullptr, nullptr, (WrWorkspace *)ws};
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(B * (D / 4), 256, 4 * kSMs);
    embloss_sumsq_kernel<LocalTabs><<<grid, 256, 0, st>>>(p, D);
    WR_CHECK_LAUNCH();
    embloss_scatter_kernel<LocalTabs><<<grid, 256, 0, st>>>(p, D);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

// Reduce this rank's inbox into its gradient shard: for every sender s and slot j, idx = inbox_idx[s][j] (0 = empty),
// G[idx - 1] += inbox_rows[s][j]; the slot is cleared for the next step.  One warp per slot, lanes over the row.
__global__ void __launch_bounds__(256) inbox_scatter_kernel(float *G, const float *__restrict__ rows, int32_t *idx,
                                                             int64_t n_slots, int D, uint32_t *touched) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int D4 = D >> 2;
    // lanes first look at 32 slots at once (most are empty: only 1/world of the senders' rows live here)
    for (int64_t base = warp * 32; base < n_slots; base += nwarps * 32) {
        const int64_t j = base + lane;
        const int32_t mine = j < n_slots ? idx[j] : 0;
        if (mine != 0) idx[j] = 0;
        uint32_t live = __ballot_sync(0xffffffffu, mine != 0);
        while (live) {
            const int src = __ffs(live) - 1;
            live &= live - 1;
            const int64_t row = (int64_t)__shfl_sync(0xffffffffu, mine, src) - 1;
            const float *r = rows + (base + src) * D;
            if (touched && lane == 0) atomicOr(touched + (row >> 5), 1u << (row & 31));
            for (int v = lane; v < D4; v += 32) red_add_v4(G + row * D + 4 * v, ldg4(r + 4 * v));
        }
    }
}

extern "C" int wr_bpr_fwd_bwd_sharded_staged(const wr_shards *host_T, const wr_shards *host_Gd,
                                             float *const host_inbox_rows[WR_MAX_WORLD],
                                             int32_t *const host_inbox_idx[WR_MAX_WORLD], int64_t cap,
                                             const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B,
                                             int64_t B_global, int D, float gamma, float grad_scale, float *loss_out,
                                             void *ws, void *stream) {
    if (!host_T || !host_Gd || !host_inbox_rows || !host_inbox_idx || !user || !pos || !neg || !loss_out || !ws)
        return WR_E_NULL;
    int rc = wr_check_shards(host_T);
    if (rc) return rc;
    rc = wr_check_shards(host_Gd);
    if (rc) return rc;
    if (B <= 0 || B_global < B || cap < 3 * B) return WR_E_SIZE;
    if (!(D == 16 || D == 32 || D == 64 || D == 128 || D == 256)) return WR_E_DIM;
    BprParamsT<StageTabs> p{{*host_T, *host_Gd, {}, {}, cap, nullptr, nullptr, nullptr}, user, pos, neg, B, host_T->n_users, host_T->n_items,
                            gamma, grad_scale / (float)B_global, (float)B_global, loss_out, 0, (WrWorkspace *)ws};
    for (int g = 0; g < host_T->world; ++g) {
        if (!host_inbox_rows[g] || !host_inbox_idx[g]) return WR_E_NULL;
        if (!wr_aligned16(host_inbox_rows[g])) return WR_E_ALIGN;
        p.tabs.inbox_rows[g] = host_inbox_rows[g];
        p.tabs.inbox_idx[g] = host_inbox_idx[g];
    }
    return launch_bpr(p, D, (cudaStream_t)stream);
}

// The same with the three rows of every batch entry already delivered by their owners (wr_xchg_request / wr_xchg_serve):
// no NVLink reads at all; gradient rows still go to the owners' inboxes.
extern "C" int wr_bpr_fwd_bwd_exchanged(const float *recv, const int32_t *where, const wr_shards *host_Gd,
                                        float *const host_inbox_rows[WR_MAX_WORLD],
                                        int32_t *const host_inbox_idx[WR_MAX_WORLD], int64_t cap, const int64_t *user,
                                        const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global, int D,
                                        float gamma, float grad_scale, uint32_t *touched, float *loss_out, void *ws,
                                        void *stream) {
    if (!recv || !where || !host_Gd || !host_inbox_rows || !host_inbox_idx || !user || !pos || !neg || !loss_out || !ws)
        return WR_E_NULL;
    const int rc = wr_check_shards(host_Gd);
    if (rc) return rc;
    if (B <= 0 || B_global < B || cap < 3 * B) return WR_E_SIZE;
    if (!(D == 16 || D == 32 || D == 64 || D == 128 || D == 256)) return WR_E_DIM;
    if (!wr_aligned16(recv)) return WR_E_ALIGN;
    BprParamsT<StageTabs> p{{*host_Gd, *host_Gd, {}, {}, cap, recv, where, touched}, user, pos, neg, B, host_Gd->n_users,
                            host_Gd->n_items, gamma, grad_scale / (float)B_global, (float)B_global, loss_out, 0,
                            (WrWorkspace *)ws};
    for (int g = 0; g < host_Gd->world; ++g) {
        if (!host_inbox_rows[g] || !host_inbox_idx[g]) return WR_E_NULL;
        if (!wr_aligned16(host_inbox_rows[g])) return WR_E_ALIGN;
        p.tabs.inbox_rows[g] = host_inbox_rows[g];
        p.tabs.inbox_idx[g] = host_inbox_idx[g];
    }
    return launch_bpr(p, D, (cudaStream_t)stream);
}

extern "C" int wr_inbox_scatter(float *G, const float *inbox_rows, int32_t *inbox_idx, int world, int64_t cap, int D,
                                void *stream) {
    return wr_inbox_scatter_marked(G, inbox_rows, inbox_idx, world, cap, D, nullptr, stream);
}

extern "C" int wr_inbox_scatter_marked(float *G, const float *inbox_rows, int32_t *inbox_idx, int world, int64_t cap,
                                       int D, uint32_t *touched, void *stream) {
    if (!G || !inbox_rows || !inbox_idx) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || cap <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(G) || !wr_aligned16(inbox_rows)) return WR_E_ALIGN;
    const int64_t n_slots = (int64_t)world * cap;
    int64_t g = (n_slots + 255) / 256;
    if (g > 16 * kSMs) g = 16 * kSMs;
    inbox_scatter_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(G, inbox_rows, inbox_idx, n_slots, D, touched);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_embloss_sumsq_sharded(const wr_shards *host_T, const int64_t *user, const int64_t *pos,
                                        const int64_t *neg, int64_t B, int D, float *sumsq_out, void *ws,
                                        void *stream) {
    if (!host_T || !user || !pos || !neg || !sumsq_out || !ws) return WR_E_NULL;
    const int rc = wr_check_shards(host_T);
    if (rc) return rc;
    if (B <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    EmbParamsT<ShardTabs> p{{*host_T, *host_T}, user, pos, neg, B, host_T->n_users, host_T->n_items, 0.f, 0.f,
                            nullptr, sumsq_out, nullptr, (WrWorkspace *)ws};
    embloss_sumsq_kernel<ShardTabs><<<grid_for(B * (D / 4), 256, 4 * kSMs), 256, 0, (cudaStream_t)stream>>>(p, D);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_embloss_scatter_sharded(const wr_shards *host_T, const wr_shards *host_Gd, const int64_t *user,
                                          const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global,
                                          int D, float reg_weight, const float *sumsq_global, float *loss_out,
                                          void *ws, void *stream) {
    if (!host_T || !host_Gd || !user || !pos || !neg || !sumsq_global || !ws) return WR_E_NULL;
    int rc = wr_check_shards(host_T);
    if (rc) return rc;
    rc = wr_check_shards(host_Gd);
    if (rc) return rc;
    if (B <= 0 || B_global < B) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    EmbParamsT<ShardTabs> p{{*host_T, *host_Gd}, user, pos, neg, B, host_T->n_users, host_T->n_items, reg_weight,
                            1.0f / (float)B_global, loss_out, nullptr, sumsq_global, (WrWorkspace *)ws};
    embloss_scatter_kernel<ShardTabs><<<grid_for(B * (D / 4), 256, 4 * kSMs), 256, 0, (cudaStream_t)stream>>>(p, D);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_adam_l2_sweep(float *P, float *M, float *V, float *G, int64_t n_elems, float l2, double beta1,
                                double beta2, float eps, float step_size, float bc2_sqrt, const float *dev_scalars,
                                void *stream) {
    if (!P || !M || !V || !G) return WR_E_NULL;
    if (n_elems <= 0) return WR_E_SIZE;
    if (!wr_aligned16(P) || !wr_aligned16(M) || !wr_aligned16(V) || !wr_aligned16(G)) return WR_E_ALIGN;
    // torch evaluates 1-beta in Python double and hands the fp32 kernels the rounded value
    AdamScalars s{l2, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), eps, step_size, bc2_sqrt};
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n4 = n_elems >> 2;
    if (n4 > 0) {
        // Large tables: 4 independent 16 B loads x 4 arrays in flight per thread, 2 CTAs/SM, whole waves.
        // Small (cache-sized) tables are latency-bound: one float4 per array per thread, as many CTAs as it takes,
        // so that every load of the sweep is issued in the first microsecond.
        if (n4 >= (int64_t)8 * kSMs * 256 * 4) {
            const int grid = grid_for(n4, 256 * 4, 8 * kSMs);
            adam_sweep_kernel<4><<<grid, 256, 0, st>>>((float4 *)P, (float4 *)M, (float4 *)V, (float4 *)G, n4, s,
                                                        dev_scalars);
        } else {
            const int grid = grid_for(n4, 256, 8 * kSMs);
            adam_sweep_kernel<1><<<grid, 256, 0, st>>>((float4 *)P, (float4 *)M, (float4 *)V, (float4 *)G, n4, s,
                                                        dev_scalars);
        }
        WR_CHECK_LAUNCH();
    }
    if (n_elems & 3) {
        adam_tail_kernel<<<1, 32, 0, st>>>(P, M, V, G, n4 << 2, n_elems, s, dev_scalars);
        WR_CHECK_LAUNCH();
    }
    return WR_OK;
}

extern "C" int wr_mark_rows(const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B, int64_t n_users,
                            int64_t n_items, uint32_t *touched, void *stream) {
    if (!user || !pos || !neg || !touched) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0) return WR_E_SIZE;
    mark_rows_kernel<<<(int)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(user, pos, neg, B, n_users, n_items, touched);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_adam_l2_sweep_marked(float *P, float *M, float *V, float *G, int64_t n_rows, int D, uint32_t *touched,
                                       float l2, double beta1, double beta2, float eps, float step_size, float bc2_sqrt,
                                       const float *dev_scalars, void *stream) {
    if (!P || !M || !V || !G || !touched) return WR_E_NULL;
    if (n_rows <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(P) || !wr_aligned16(M) || !wr_aligned16(V) || !wr_aligned16(G)) return WR_E_ALIGN;
    AdamScalars s{l2, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), eps, step_size, bc2_sqrt};
    cudaStream_t st = (cudaStream_t)stream;
    const int D4 = D >> 2;
    int shift = -1;
    if ((D4 & (D4 - 1)) == 0) {
        shift = 0;
        while ((1 << shift) < D4) ++shift;
    }
    const int64_t n4 = n_rows * D4;
    if (n4 >= (int64_t)8 * kSMs * 256 * 4) {
        const int grid = grid_for(n4, 256 * 4, 8 * kSMs);
        adam_sweep_marked_kernel<4><<<grid, 256, 0, st>>>((float4 *)P, (float4 *)M, (float4 *)V, (float4 *)G, n4, D4, shift,
                                                           touched, s, dev_scalars);
    } else {
        const int grid = grid_for(n4, 256, 8 * kSMs);
        adam_sweep_marked_kernel<1><<<grid, 256, 0, st>>>((float4 *)P, (float4 *)M, (float4 *)V, (float4 *)G, n4, D4, shift,
                                                           touched, s, dev_scalars);
    }
    WR_CHECK_LAUNCH();
    // every bit goes back to zero behind the sweep (stream order): the next step's markers start from a clean map
    const cudaError_t e = cudaMemsetAsync(touched, 0, (size_t)((n_rows + 31) / 32) * sizeof(uint32_t), st);
    return e == cudaSuccess ? WR_OK : (int)e;
}

// Largest grid of bprmf_step_kernel<...>: one CTA per SM (up to 1,024 threads each), at most WR_EP_MAX_GRID arrival
// lines (cached per instantiation).
template <int LPR, int VPL, class TABS>
static int step_max_grid(int *out) {
    static int cached = 0;
    if (!cached) {
        int dev = 0, sms = 0, per_sm = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess)
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bprmf_step_kernel<LPR, VPL, TABS>, 1024, 0);
        if (e != cudaSuccess) return (int)e;
        if (per_sm < 1) return (int)cudaErrorLaunchOutOfResources;
        cached = sms < WR_EP_MAX_GRID ? sms : WR_EP_MAX_GRID;
    }
    *out = cached;
    return 0;
}

static bool g_step_trace_on = false;      // wr_debug_step_trace: one-GPU launches take the TRACE instantiation

template <int LPR, int VPL, class TABS>
static int launch_step_fused(BprParamsT<TABS> &bp, float *P, float *M, float *V, float *G, int64_t n4, AdamScalars &s,
                             const float *dev_scalars, StepSync &sy, cudaStream_t st) {
    int max_grid = 0;
    const int rc = step_max_grid<LPR, VPL, TABS>(&max_grid);
    if (rc) return rc;
    // Every thread updates `per` float4 of each array (even: the Adam loop keeps two in flight), as few as 1,024-thread
    // CTAs on every SM allow; then the fewest threads per CTA (whole warps) and the fewest CTAs for that share.  The bench
    // shape (155,936 float4 per array, 148 SMs): per = 2, 544 threads, 144 CTAs.
    const int64_t per = 2 * ((n4 + 2048 * (int64_t)max_grid - 1) / (2048 * (int64_t)max_grid));
    const int threads = (int)((n4 + max_grid * per - 1) / (max_grid * per) + 31) / 32 * 32;
    const int grid = grid_for(n4, (int)(threads * per), max_grid);
    float4 *P4 = (float4 *)P, *M4 = (float4 *)M, *V4 = (float4 *)V, *G4 = (float4 *)G;
    void *args[] = {&bp, &P4, &M4, &V4, &G4, &n4, &s, &dev_scalars, &sy};
    const void *fn = (const void *)bprmf_step_kernel<LPR, VPL, TABS>;
    if constexpr (std::is_same<TABS, LocalTabs>::value && VPL == 1)      // D <= 128 (D = 256 would spill with the stamps)
        if (g_step_trace_on) fn = (const void *)bprmf_step_kernel<LPR, VPL, TABS, true>;
    return (int)cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(threads), args, 0, st);
}

template <class TABS>
static int dispatch_step_fused(BprParamsT<TABS> &bp, int D, float *P, float *M, float *V, float *G, int64_t n4,
                               AdamScalars &s, const float *dev_scalars, StepSync &sy, cudaStream_t st) {
    switch (D) {
        case 16: return launch_step_fused<4, 1, TABS>(bp, P, M, V, G, n4, s, dev_scalars, sy, st);
        case 32: return launch_step_fused<8, 1, TABS>(bp, P, M, V, G, n4, s, dev_scalars, sy, st);
        case 64: return launch_step_fused<16, 1, TABS>(bp, P, M, V, G, n4, s, dev_scalars, sy, st);
        case 128: return launch_step_fused<32, 1, TABS>(bp, P, M, V, G, n4, s, dev_scalars, sy, st);
        case 256: return launch_step_fused<32, 2, TABS>(bp, P, M, V, G, n4, s, dev_scalars, sy, st);
        default: return WR_E_DIM;
    }
}

// Tables up to this many bytes per array take the single-launch step (they fit in L2 several times over and the
// step is bound by launch / DRAM latency); larger ones stream at HBM bandwidth through the two-kernel path.
#define WR_FUSED_STEP_MAX_ELEMS ((int64_t)8 << 20)

extern "C" int wr_bprmf_step(float *P, float *M, float *V, float *G, const int64_t *user, const int64_t *pos,
                             const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items, float gamma,
                             float l2, double beta1, double beta2, float eps, float step_size, float bc2_sqrt,
                             const float *dev_scalars, float *loss_out, void *ws, void *stream) {
    if (!P || !M || !V || !G || !user || !pos || !neg || !loss_out || !ws) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0 || n_users >= INT32_MAX || n_items >= INT32_MAX) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(P) || !wr_aligned16(M) || !wr_aligned16(V) || !wr_aligned16(G)) return WR_E_ALIGN;
    return wr_bprmf_step_impl(P, M, V, G, user, pos, neg, B, D, n_users, n_items, gamma, l2, beta1, beta2, eps, step_size,
                              bc2_sqrt, dev_scalars, loss_out, ws, stream);
}

// wr_bprmf_step with a row map for the streaming (two-kernel) path: the batch's rows are marked, the gradient kernel
// accumulates into them and the sweep reads G only where a bit is set.  Cache-sized tables take the single launch and
// leave the map alone.  Results are those of wr_bprmf_step bit for bit (a skipped G row held zeros).
extern "C" int wr_bprmf_step_marked(float *P, float *M, float *V, float *G, uint32_t *touched, const int64_t *user,
                                    const int64_t *pos, const int64_t *neg, int64_t B, int D, int64_t n_users,
                                    int64_t n_items, float gamma, float l2, double beta1, double beta2, float eps,
                                    float step_size, float bc2_sqrt, const float *dev_scalars, float *loss_out, void *ws,
                                    void *stream) {
    if (!P || !M || !V || !G || !touched || !user || !pos || !neg || !loss_out || !ws) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0 || n_users >= INT32_MAX || n_items >= INT32_MAX) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(P) || !wr_aligned16(M) || !wr_aligned16(V) || !wr_aligned16(G)) return WR_E_ALIGN;
    const int64_t n_elems = (n_users + n_items) * D;
    const bool fused_shape = D == 16 || D == 32 || D == 64 || D == 128 || D == 256;
    if (fused_shape && n_elems <= WR_FUSED_STEP_MAX_ELEMS)
        return wr_bprmf_step_impl(P, M, V, G, user, pos, neg, B, D, n_users, n_items, gamma, l2, beta1, beta2, eps,
                                  step_size, bc2_sqrt, dev_scalars, loss_out, ws, stream);
    int rc = wr_mark_rows(user, pos, neg, B, n_users, n_items, touched, stream);
    if (rc) return rc;
    rc = wr_bpr_fwd_bwd(P, P + n_users * D, user, pos, neg, B, D, n_users, n_items, gamma, 1.0f, G, G + n_users * D,
                        loss_out, 0, ws, stream);
    if (rc) return rc;
    return wr_adam_l2_sweep_marked(P, M, V, G, n_users + n_items, D, touched, l2, beta1, beta2, eps, step_size, bc2_sqrt,
                                   dev_scalars, stream);
}

// The per-step launches: one cooperative launch (parameter loads first, BPR, grid barrier, Adam) for tables of up to
// 8 Mi elements, two kernels beyond that.
int wr_bprmf_step_impl(float *P, float *M, float *V, float *G, const int64_t *user, const int64_t *pos,
                       const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items, float gamma, float l2,
                       double beta1, double beta2, float eps, float step_size, float bc2_sqrt, const float *dev_scalars,
                       float *loss_out, void *ws, void *stream) {
    const int64_t n_elems = (n_users + n_items) * D;
    const bool fused_shape = D == 16 || D == 32 || D == 64 || D == 128 || D == 256;
    if (!fused_shape || n_elems > WR_FUSED_STEP_MAX_ELEMS) {
        int rc = wr_bpr_fwd_bwd(P, P + n_users * D, user, pos, neg, B, D, n_users, n_items, gamma, 1.0f, G,
                                G + n_users * D, loss_out, 0, ws, stream);
        if (rc) return rc;
        return wr_adam_l2_sweep(P, M, V, G, n_elems, l2, beta1, beta2, eps, step_size, bc2_sqrt, dev_scalars, stream);
    }
    BprParams bp{{P, P + n_users * D, G, G + n_users * D}, user, pos, neg, B, n_users, n_items, gamma,
                 1.0f / (float)B, (float)B, loss_out, 0, (WrWorkspace *)ws};
    AdamScalars s{l2, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), eps, step_size, bc2_sqrt};
    StepSync sy{};
    sy.world = 1;
    return dispatch_step_fused(bp, D, P, M, V, G, n_elems >> 2, s, dev_scalars, sy, (cudaStream_t)stream);
}

extern "C" int wr_debug_step_trace(uint64_t *dev_trace) {
    const cudaError_t e = cudaMemcpyToSymbol(g_step_trace, &dev_trace, sizeof(dev_trace));
    if (e != cudaSuccess) return (int)e;
    g_step_trace_on = dev_trace != nullptr;
    return WR_OK;
}

extern "C" int wr_bprmf_step_sharded_supported(int64_t n_local_rows, int D) {
    const bool fused_shape = D == 16 || D == 32 || D == 64 || D == 128 || D == 256;
    return fused_shape && n_local_rows > 0 && n_local_rows * D <= WR_FUSED_STEP_MAX_ELEMS;
}

extern "C" int wr_bprmf_step_sharded(const wr_shards *host_T, const wr_shards *host_Gd, float *M, float *V,
                                     const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B,
                                     int64_t B_global, int D, float gamma, float l2, double beta1, double beta2,
                                     float eps, float step_size, float bc2_sqrt, uint32_t epoch,
                                     uint32_t *const host_flags[WR_MAX_WORLD], float *const host_slots[WR_MAX_WORLD],
                                     float *loss_out, void *ws, void *stream) {
    if (!host_T || !host_Gd || !M || !V || !user || !pos || !neg || !host_flags || !host_slots || !loss_out || !ws)
        return WR_E_NULL;
    int rc = wr_check_shards(host_T);
    if (rc) return rc;
    rc = wr_check_shards(host_Gd);
    if (rc) return rc;
    if (B <= 0 || B_global < B || epoch == 0) return WR_E_SIZE;
    const int64_t n_local = host_T->rows_u_local + host_T->rows_i_local;
    if (!wr_bprmf_step_sharded_supported(n_local, D)) return WR_E_DIM;
    if (!wr_aligned16(M) || !wr_aligned16(V)) return WR_E_ALIGN;
    StepSync sy{};
    sy.world = host_T->world;
    sy.rank = host_T->rank;
    sy.epoch = epoch;
    for (int g = 0; g < sy.world; ++g) {
        if (!host_flags[g] || !host_slots[g]) return WR_E_NULL;
        sy.flags[g] = host_flags[g];
        sy.slots[g] = host_slots[g];
    }
    BprParamsT<ShardTabs> bp{{*host_T, *host_Gd}, user, pos, neg, B, host_T->n_users, host_T->n_items, gamma,
                             1.0f / (float)B_global, (float)B_global, loss_out, 0, (WrWorkspace *)ws};
    AdamScalars s{l2, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), eps, step_size, bc2_sqrt};
    float *P = host_T->base[host_T->rank], *G = host_Gd->base[host_Gd->rank];
    return dispatch_step_fused(bp, D, P, M, V, G, (n_local * D) >> 2, s, nullptr, sy, (cudaStream_t)stream);
}

extern "C" int wr_bprmf_step_host(const int64_t *host_ids, int64_t *dev_ids, float *host_loss, float *P, float *M,
                                  float *V, float *G, int64_t B, int D, int64_t n_users, int64_t n_items,
                                  float gamma, float l2, double beta1, double beta2, float eps, float step_size,
                                  float bc2_sqrt, float *loss_out, void *ws, void *stream, int sync) {
    if (!host_ids || !dev_ids || !host_loss) return WR_E_NULL;
    if (B <= 0) return WR_E_SIZE;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(dev_ids, host_ids, (size_t)(3 * B) * sizeof(int64_t), cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return (int)e;
    const int rc = wr_bprmf_step(P, M, V, G, dev_ids, dev_ids + B, dev_ids + 2 * B, B, D, n_users, n_items, gamma, l2,
                                 beta1, beta2, eps, step_size, bc2_sqrt, nullptr, loss_out, ws, stream);
    if (rc) return rc;
    e = cudaMemcpyAsync(host_loss, loss_out, sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return (int)e;
    if (sync) e = cudaStreamSynchronize(st);
    return (int)e;
}

extern "C" int wr_gather_rows(const float *T, const int64_t *idx, int64_t B, int D, int64_t n_rows, float *out,
                              void *ws, void *stream) {
    if (!T || !idx || !out || !ws) return WR_E_NULL;
    if (B < 0 || n_rows <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(T) || !wr_aligned16(out)) return WR_E_ALIGN;
    if (B == 0) return WR_OK;
    gather_rows_kernel<<<grid_for(B * (D / 4), 256, 8 * kSMs), 256, 0, (cudaStream_t)stream>>>(
        T, idx, B, D, n_rows, out, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_scatter_add_rows(float *G, const int64_t *idx, int64_t B, int D, int64_t n_rows,
                                   const float *rows, void *ws, void *stream) {
    if (!G || !idx || !rows || !ws) return WR_E_NULL;
    if (B < 0 || n_rows <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(G) || !wr_aligned16(rows)) return WR_E_ALIGN;
    if (B == 0) return WR_OK;
    scatter_add_rows_kernel<<<grid_for(B * (D / 4), 256, 8 * kSMs), 256, 0, (cudaStream_t)stream>>>(
        G, idx, B, D, n_rows, rows, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    return WR_OK;
}
