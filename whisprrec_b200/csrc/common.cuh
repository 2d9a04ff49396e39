// Shared device helpers for libwhisprrec_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/whisprrec_b200.h"

#define WR_MAX_PARTIAL_BLOCKS 2048
#define WR_EP_PART_DEPTH 4      // steps whose per-CTA loss partials may be waiting for their reduction
#define WR_EP_MAX_GRID 256      // CTAs of the resident kernel (one per SM)

// Device scratch block handed in by the caller (wr_workspace_bytes()).
struct WrWorkspace {
    uint32_t status;                           // WR_STATUS_* bits
    uint32_t ticket[7];                        // "last block done" counters, one per reduction in flight
    float norms[4];                            // EmbLoss: ||U0_b||, ||P0_b||, ||N0_b||
    float partial[3 * WR_MAX_PARTIAL_BLOCKS];  // per-block partial sums, summed in block order (deterministic)
    double dpartial[2 * 8 * 64];               // wr_metrics
    // ---- resident BPRMF kernel (epoch_kernel.cu); every word is left zero by the last CTA to leave ----
    uint32_t ep_pad0;
    uint32_t ep_pad1;
    uint32_t ep_abort;                         // a wait gave up: every CTA leaves
    uint32_t ep_depart;                        // departures (workers + helper of every CTA)
    uint32_t ep_loss_flag[WR_EP_PART_DEPTH];   // step + 1 of the last loss reduced out of each partial slot
    float ep_partial[WR_EP_PART_DEPTH * WR_EP_MAX_GRID];
    uint32_t ep_fetched[16];                   // streaming: helper warps that have copied their piece of step s's ids, at
                                               // [(s - first) % 16]; cumulative per slot (helpers run < 16 steps apart)
    uint32_t ep_flag[WR_EP_MAX_GRID * 32];     // grid barrier: CTA c's arrival number at [32 c] (one 128-byte line each)
    // ---- single-launch step (bprmf_step_kernel); never reset: both words only move forward ----
    uint32_t st_gen;                           // grid barrier generation: launches so far
    uint32_t st_pad[31];
    uint32_t st_flag[WR_EP_MAX_GRID * 32];     // CTA c's arrival (generation + 1) at [32 c]
};

#define WR_CHECK_LAUNCH()                        \
    do {                                         \
        cudaError_t e__ = cudaGetLastError();    \
        if (e__ != cudaSuccess) return (int)e__; \
    } while (0)

int wr_check_shards(const wr_shards *s);   // train_kernels.cu

static inline bool wr_aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

namespace wr {

// SMs of the current device (148 on a B200), asked once per translation unit: grids are sized in multiples of it.
static inline int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}
#define kSMs (::wr::sm_count())

// ---- top-k lists with k up to 256 (wr_eval_rank_topk_long, DESIGN.md section 4.3) ----
constexpr int WR_LONG_KMAX = 256;
constexpr int WR_LONG_SEG_CAP = 4096;            // candidate ids kept per row; a row with more is finished by a sweep
constexpr int WR_LONG_RANGES = 16;               // item ranges of the bound pass: ceil(k / 32) .. 2 ceil(k / 32) - 1
constexpr int64_t WR_LONG_BLOCK_ROWS = 65536;    // rows per block, so that the segments stay <= 1 GB

// The part of a long call's scratch that both precisions use: a 1,024-byte header at offset 0 (word 0: rows the sweep
// finished, read by the caller), then -- after precision 2's tensor-core scratch -- these per-row-block arrays.
struct LongScratch {
    float *bound;        // [rows][WR_LONG_RANGES] the k'-th best score of each item range
    int32_t *seg_cnt;    // [rows] candidates appended
    int32_t *seg;        // [rows][WR_LONG_SEG_CAP] candidate item ids
    static size_t align(size_t x) { return (x + 1023) / 1024 * 1024; }
    static size_t bytes(int64_t rows) {
        return align((size_t)rows * WR_LONG_RANGES * 4) + align((size_t)rows * 4) + (size_t)rows * WR_LONG_SEG_CAP * 4;
    }
    LongScratch(void *base, int64_t rows) {
        uint8_t *p = static_cast<uint8_t *>(base);
        bound = reinterpret_cast<float *>(p);
        seg_cnt = reinterpret_cast<int32_t *>(p + align((size_t)rows * WR_LONG_RANGES * 4));
        seg = reinterpret_cast<int32_t *>(p + align((size_t)rows * WR_LONG_RANGES * 4) + align((size_t)rows * 4));
    }
};

// The select pass of a long call (eval_kernels.cu): one CTA per row re-scores the row's candidates with precision 0's FMA
// chain and sorts them by (value desc, id asc); a row whose segment overflowed is swept over every item instead.
struct LongSelect {
    const int32_t *seg, *seg_cnt;
    int64_t R;                   // rows of this block
    const float *U;              // user table (rows_gathered = 0: row r is U[user[r]]) or the block's gathered rows
    const int64_t *user;
    int rows_gathered;
    const float *I;
    int D;
    int64_t n_items;
    const int64_t *hist_ptr;
    const int32_t *hist_idx;
    int k;
    int32_t *topk_idx;           // the block's [R][k] outputs
    float *topk_val;
    uint32_t *fallback;          // rows swept (header word 0 of the scratch)
    uint32_t *status;
};
int long_select(const LongSelect &q, cudaStream_t st);

// Item ranges of the bound pass over n_tiles tiles for a k-list: need = ceil(k / 32) or more ranges of whole tiles (the
// last may be short), each giving the k'-th best of its items, k' = ceil(k / need) <= 32, from the k <= 32 list
// machinery.  Returns the number of ranges (0: fewer tiles than need -- no bound, every unmasked item is a candidate) and
// sets the tiles per range, k' and need.
static inline int long_ranges(int n_tiles, int k, int *tiles_per_range, int *kp, int *need) {
    *need = (k + 31) / 32;
    *kp = (k + *need - 1) / *need;
    if (n_tiles < *need) return 0;
    *tiles_per_range = n_tiles / *need;
    return (n_tiles + *tiles_per_range - 1) / *tiles_per_range;      // need .. 2 need - 1
}

// The collect pass's threshold for one row: the need-th largest of its n range bounds b.  The need ranges whose bounds
// are at least that large each hold k' unmasked items scoring at or above their bound, so need k' >= k items reach it: a
// lower bound on the row's k-th best.  -inf when fewer than need ranges hold k' items (or n = 0).
__device__ __forceinline__ float long_bound(const float *b, int n, int need) {
    float L = -INFINITY;
    for (int c = 0; c < n; ++c) {
        int ge = 0;
        for (int c2 = 0; c2 < n; ++c2) ge += b[c2] >= b[c] ? 1 : 0;
        if (ge >= need) L = fmaxf(L, b[c]);
    }
    return L;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int WIDTH>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum over the block; the result is valid in thread 0.  `red` needs blockDim.x/32 floats.
__device__ __forceinline__ float block_sum(float v, float *red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    float t = 0.f;
    if (w == 0) {
        t = lane < nw ? red[lane] : 0.f;
        t = warp_sum(t);
    }
    return t;
}

// 128-bit fire-and-forget reduction into global memory (REDG.E.ADD.F32x4): one L2 transaction per 16 B.
__device__ __forceinline__ void red_add_v4(float *addr, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

__device__ __forceinline__ uint64_t global_timer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 scale4(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ float4 sub4(float4 a, float4 b) {
    return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
}
__device__ __forceinline__ float4 add4(float4 a, float4 b) {
    return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 fma4(float s, float4 x, float4 a) {
    return make_float4(fmaf(s, x.x, a.x), fmaf(s, x.y, a.y), fmaf(s, x.z, a.z), fmaf(s, x.w, a.w));
}

// ---- pointwise math shared by the step kernels ----
__device__ __forceinline__ void bpr_pointwise(float sp, float sn, float gamma, float coef, float &loss, float &c) {
    // utils/loss.py:38: -log(gamma + sigmoid(pos - neg)); d/ds+ = -(sig (1-sig)) / (gamma + sig)
    const float x = sp - sn;
    if (gamma < 0.f) {
        // SGL.py:183: -logsigmoid(x) = softplus(-x) = max(-x, 0) + log1p(exp(-|x|)); d/dx = -sigmoid(-x)
        const float e = expf(-fabsf(x));
        loss = fmaxf(-x, 0.f) + log1pf(e);
        c = -(x >= 0.f ? e / (1.0f + e) : 1.0f / (1.0f + e)) * coef;
        return;
    }
    const float sig = 1.0f / (1.0f + expf(-x));
    loss = -logf(gamma + sig);
    c = -(sig * (1.0f - sig)) / (gamma + sig) * coef;
}

struct AdamScalars {
    float l2, w1, beta2, w2, eps, step_size, bc2_sqrt;
};

__device__ __forceinline__ void adam_elem(float &p, float &m, float &v, float g, const AdamScalars &s) {
    g = fmaf(s.l2, p, g);                    // grad.add(param, alpha=weight_decay)
    m = fmaf(s.w1, g - m, m);                // exp_avg.lerp_(grad, 1 - beta1)
    v = fmaf(s.w2 * g, g, v * s.beta2);      // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    const float denom = sqrtf(v) / s.bc2_sqrt + s.eps;
    p = p + (-s.step_size * m) / denom;      // param.addcdiv_(exp_avg, denom, value=-step_size)
}

// ~1 ulp quotient / square root from the MUFU approximations plus one Newton step: the IEEE sequences of `/` and sqrtf
// cost ~25 instructions each, which makes a cache-resident Adam phase issue-bound (scripts/prof_resident.py).
__device__ __forceinline__ float div_nr(float n, float d) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
    const float q = n * r;
    return fmaf(fmaf(-d, q, n), r, q);
}
__device__ __forceinline__ float sqrt_nr(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    const float s = x * r;
    const float t = fmaf(fmaf(-s, s, x), 0.5f * r, s);
    return x > 1e-37f ? t : 0.f;             // 0 (r = inf) and denormals
}
// adam_elem with div_nr / sqrt_nr and the bias-correction division folded into a multiplication (inv_bc2 = 1 / bc2_sqrt)
__device__ __forceinline__ void adam_elem_nr(float &p, float &m, float &v, float g, const AdamScalars &s, float inv_bc2) {
    g = fmaf(s.l2, p, g);
    m = fmaf(s.w1, g - m, m);
    v = fmaf(s.w2 * g, g, v * s.beta2);
    const float denom = fmaf(sqrt_nr(v), inv_bc2, s.eps);
    p = p + div_nr(-s.step_size * m, denom);
}

// ---- scoped loads / stores for the in-kernel meeting points ----
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint32_t ld_relaxed_gpu_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// The last block to arrive returns true (after all other blocks' prior global writes are visible).
__device__ __forceinline__ bool last_block_arrives(uint32_t *ticket, bool *smem_flag) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const uint32_t t = atomicAdd(ticket, 1u);
        *smem_flag = (t == gridDim.x - 1);
        if (*smem_flag) *ticket = 0;  // re-arm for the next launch on this stream
    }
    __syncthreads();
    const bool last = *smem_flag;
    if (last) __threadfence();
    return last;
}

// Row layout shared by the gather-style kernels: a row of D = 4*LPR*VPL floats is covered by LPR lanes,
// each holding VPL float4 at stride LPR; 32/LPR rows are processed by a warp at a time.
template <int LPR, int VPL>
struct RowGroup {
    static constexpr int D = 4 * LPR * VPL;
    static constexpr int GROUPS = 32 / LPR;
    __device__ static __forceinline__ void load(const float *row, int sub, float4 (&r)[VPL]) {
#pragma unroll
        for (int v = 0; v < VPL; ++v) r[v] = ldg4(row + 4 * (sub + v * LPR));
    }
    // tables that the same kernel (or a peer) rewrites: read through L2, never the non-coherent path
    __device__ static __forceinline__ void load_cg(const float *row, int sub, float4 (&r)[VPL]) {
#pragma unroll
        for (int v = 0; v < VPL; ++v) r[v] = __ldcg(reinterpret_cast<const float4 *>(row + 4 * (sub + v * LPR)));
    }
    __device__ static __forceinline__ void zero(float4 (&r)[VPL]) {
#pragma unroll
        for (int v = 0; v < VPL; ++v) r[v] = f4_zero();
    }
};

// ---- where a table row lives: one GPU, or the cyclic row shards of a multi-GPU job reached through peer memory ----
struct LocalTabs {
    const float *U, *I;
    float *gU, *gI;
    __device__ __forceinline__ const float *urow(int64_t u, int D) const { return U + u * D; }
    __device__ __forceinline__ const float *irow(int64_t i, int D) const { return I + i * D; }
    // row of batch entry b in role `which` (0 user, 1 positive, 2 negative) whose id is `id`
    __device__ __forceinline__ const float *row(int64_t, int which, int64_t id, int D) const {
        return (which == 0 ? U : I) + id * D;
    }
    __device__ __forceinline__ float *gurow(int64_t u, int D) const { return gU + u * D; }
    __device__ __forceinline__ float *girow(int64_t i, int D) const { return gI + i * D; }
    // gradient contribution `v` to floats [off, off+4) of a row; (b, which) name the batch row and its role
    __device__ __forceinline__ void add_user(int64_t u, int D, int off, float4 v, int64_t, int) const {
        red_add_v4(gU + u * D + off, v);
    }
    __device__ __forceinline__ void add_item(int64_t i, int D, int off, float4 v, int64_t, int) const {
        red_add_v4(gI + i * D + off, v);
    }
};

// user u -> rank u % world, local row u / world; item i -> rank i % world, local row rows_u_local + i / world.
// Ids are < 2^31 (checked on the host), so the divisions are 32-bit.
__device__ __forceinline__ float *shard_user_row(const wr_shards &s, int64_t u, int D) {
    const uint32_t q = (uint32_t)u / (uint32_t)s.world, r = (uint32_t)u - q * (uint32_t)s.world;
    return s.base[r] + (int64_t)q * D;
}
__device__ __forceinline__ float *shard_item_row(const wr_shards &s, int64_t i, int D) {
    const uint32_t q = (uint32_t)i / (uint32_t)s.world, r = (uint32_t)i - q * (uint32_t)s.world;
    return s.base[r] + (s.rows_u_local + (int64_t)q) * D;
}
__device__ __forceinline__ float *shard_node_row(const wr_shards &s, int64_t n, int D) {
    return n < s.n_users ? shard_user_row(s, n, D) : shard_item_row(s, n - s.n_users, D);
}

struct ShardTabs {
    wr_shards t, g;
    __device__ __forceinline__ const float *urow(int64_t u, int D) const { return shard_user_row(t, u, D); }
    __device__ __forceinline__ const float *irow(int64_t i, int D) const { return shard_item_row(t, i, D); }
    __device__ __forceinline__ const float *row(int64_t, int which, int64_t id, int D) const {
        return which == 0 ? shard_user_row(t, id, D) : shard_item_row(t, id, D);
    }
    __device__ __forceinline__ float *gurow(int64_t u, int D) const { return shard_user_row(g, u, D); }
    __device__ __forceinline__ float *girow(int64_t i, int D) const { return shard_item_row(g, i, D); }
    __device__ __forceinline__ void add_user(int64_t u, int D, int off, float4 v, int64_t, int) const {
        red_add_v4(shard_user_row(g, u, D) + off, v);       // remote rows: a reduction over NVLink per 16 bytes
    }
    __device__ __forceinline__ void add_item(int64_t i, int D, int off, float4 v, int64_t, int) const {
        red_add_v4(shard_item_row(g, i, D) + off, v);
    }
};

// Large batches: 16-byte reductions over NVLink do not scale (every one is its own fabric transaction).  Remote
// gradient rows are instead WRITTEN (plain coalesced stores) into the owner's inbox -- slot 3 b + which of the
// sender's region, no counters, no atomics -- together with the owner-local row index (+1; 0 = empty), and the owner
// reduces its inbox into its gradient shard locally after the barrier (inbox_scatter_kernel).
struct StageTabs {
    wr_shards t, g;
    float *inbox_rows[WR_MAX_WORLD];     // rank o's [world][cap][D]
    int32_t *inbox_idx[WR_MAX_WORLD];    // rank o's [world][cap]
    int64_t cap;                         // slots per sender (>= 3 x the largest per-rank batch)
    // rows already delivered by their owners (wr_xchg_*): batch entry b's row in role `which` is recv[where[3 b + which]]
    const float *recv;
    const int32_t *where;
    uint32_t *touched;                   // nullable: bitmap over this rank's rows, set for rows reduced in place
    __device__ __forceinline__ const float *urow(int64_t u, int D) const { return shard_user_row(t, u, D); }
    __device__ __forceinline__ const float *irow(int64_t i, int D) const { return shard_item_row(t, i, D); }
    __device__ __forceinline__ const float *row(int64_t b, int which, int64_t id, int D) const {
        if (recv) return recv + (int64_t)where[3 * b + which] * D;
        return which == 0 ? shard_user_row(t, id, D) : shard_item_row(t, id, D);
    }
    __device__ __forceinline__ float *gurow(int64_t u, int D) const { return shard_user_row(g, u, D); }
    __device__ __forceinline__ float *girow(int64_t i, int D) const { return shard_item_row(g, i, D); }
    __device__ __forceinline__ void put(uint32_t owner, int64_t local_row, int D, int off, float4 v, int64_t b,
                                        int which) const {
        if ((int)owner == g.rank) {
            red_add_v4(g.base[owner] + local_row * D + off, v);
            if (touched && off == 0) atomicOr(touched + (local_row >> 5), 1u << (local_row & 31));
            return;
        }
        const int64_t slot = (int64_t)g.rank * cap + 3 * b + which;
        *reinterpret_cast<float4 *>(inbox_rows[owner] + slot * D + off) = v;
        if (off == 0) inbox_idx[owner][slot] = (int32_t)local_row + 1;
    }
    __device__ __forceinline__ void add_user(int64_t u, int D, int off, float4 v, int64_t b, int which) const {
        const uint32_t q = (uint32_t)u / (uint32_t)g.world, r = (uint32_t)u - q * (uint32_t)g.world;
        put(r, (int64_t)q, D, off, v, b, which);
    }
    __device__ __forceinline__ void add_item(int64_t i, int D, int off, float4 v, int64_t b, int which) const {
        const uint32_t q = (uint32_t)i / (uint32_t)g.world, r = (uint32_t)i - q * (uint32_t)g.world;
        put(r, g.rows_u_local + (int64_t)q, D, off, v, b, which);
    }
};

}  // namespace wr

// Dispatch on the embedding size: the row is split over LPR lanes x VPL float4 per lane.
#define WR_DISPATCH_D(D, CALL)                 \
    switch (D) {                               \
        case 4: { CALL(1, 1); } break;         \
        case 8: { CALL(2, 1); } break;         \
        case 16: { CALL(4, 1); } break;        \
        case 32: { CALL(8, 1); } break;        \
        case 64: { CALL(16, 1); } break;       \
        case 128: { CALL(32, 1); } break;      \
        case 256: { CALL(32, 2); } break;      \
        case 512: { CALL(32, 4); } break;      \
        default: return WR_E_DIM;              \
    }
