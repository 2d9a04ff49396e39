// Full-ranking evaluation on the 5th-generation tensor cores (precision = 1).
//
//   S[128 x 256 tile] = U_bf16[rows, D] . I_bf16[items, D]^T     tcgen05.mma, cta_group::1, M=128 N=256 K=16,
//                                                                fp32 accumulators in TMEM (2 x 256 columns)
// A CTA owns 128 eval rows and walks the item tiles in ascending order.  Warp roles:
//   warp 0      TMA producer  (A once, then a ring of B stages; SWIZZLE_128B boxes of 64 bf16 = 128 B rows)
//   warp 1      MMA issuer    (one elected lane; smem descriptors advanced 32 B per K=16 step)
//   warp 2      TMEM allocator / deallocator
//   warps 4-19  epilogue: tcgen05.ld 32 columns at a time, history mask from the sorted per-user CSR (one cursor
//               per row, the tiles arrive in item order), count of items beating the target -- while the MMA of
//               the next tile fills the other accumulator.  The score matrix never leaves TMEM.
//   warps 20-23 (top-k launches only) drain the per-row candidate rings the epilogue warps push into, keep each
//               row's k best and publish its threshold.
// precision 1: operands are rounded to bf16 once per evaluation (pack kernels below); the target score is the fp32 FMA
// chain over the same bf16-rounded operands.  Parity with the fp32 path is therefore "looser": see tests.
// precision 2 ("exact"): every fp32 operand is split into two bf16 terms, a = hi + lo, and the tensor cores accumulate
// hi.hi + hi.lo + lo.hi (K = 3 D: A' = [hi | hi | lo], B' = [hi | lo | hi]; at D = 256 only [hi | lo] of A' is stored and
// resident, the MMAs of the middle K third read its hi blocks again).  The result is within
// eps_r = c_D * ||a_r|| * max_j ||b_j|| of the fp32 FMA chain precision 0 computes (bound below), so a score farther than
// eps_r from the row's target decides the comparison as precision 0 would; the few pairs inside the band go to a
// candidate list and are re-scored with exactly precision 0's FMA chain (eval_recheck_kernel).  Ranks are therefore
// IDENTICAL to precision 0 -- the reference's fp32 ranking semantics on the tensor cores.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cstdlib>

#include "common.cuh"

namespace wr {

struct TcParams {
    const int64_t *user, *pos;
    int64_t R, n_users, n_items;
    const int64_t *hist_ptr;
    const int32_t *hist_idx;
    const float *target;        // [R] target scores (written by pack_users_kernel)
    const uint8_t *row_ok;      // [R] 1 if the row's ids were in range
    int32_t *rank;
    float *scores;              // optional dense [R, n_items] dump of the tensor-core scores (tests)
    int splits, tiles_per_split, n_tiles;
    int k;                      // top-k lists (TOPK instantiation only)
    int top_trigger;
    int32_t *topk_idx;
    float *topk_val;
    // precision 2
    const float *anorm;         // [R] ||a_r||_2 of the fp32 user rows
    const float *bmax;          // [1] max_j ||b_j||_2 of the fp32 item rows
    float band_c;               // eps_r = band_c * anorm[r] * bmax[0]
    uint2 *cand;                // (row, item) pairs inside the band
    unsigned long long *cand_cnt;
    unsigned long long cand_cap;
    uint32_t *status;           // WR_STATUS_EVAL_OVERFLOW when the list is full
    int32_t *seg;               // top-k: [rows][TC_SEG_CAP] list candidates (item ids) per row
    int32_t *seg_cnt;           // top-k: [rows] candidates appended (> TC_SEG_CAP: the segment overflowed)
    float *bound;               // long lists: [rows][WR_LONG_RANGES] the k'-th best t of each item range
    int n_bounds, bound_need;   // long lists, collect pass: ranges written by the bound pass (0: no bound), long_bound
};

constexpr int TC_KMAX = 32;
constexpr int TC_SEG_CAP = 1024;        // list candidates kept per row (precision 2 with top-k)

// ---------------------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(const CUtensorMap *map, uint64_t *bar, void *dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// K-major operand tile, 128-byte rows, SWIZZLE_128B: 8-row groups are 1024 B apart (SBO), LBO unused.
__device__ __forceinline__ uint64_t umma_desc_sw128(const void *smem) {
    const uint32_t addr = smem_u32(smem);
    uint64_t d = (uint64_t)((addr & 0x3FFFFu) >> 4);   // start address, bits [0,14)
    d |= (uint64_t)(1024u >> 4) << 32;                  // stride byte offset, bits [32,46)
    d |= 1ull << 46;                                    // descriptor version (Blackwell)
    d |= 2ull << 61;                                    // layout: SWIZZLE_128B
    return d;
}
// kind::f16, A = B = bf16, D = fp32, both K-major, M x N as given.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------------------
// operand packing: fp32 tables -> bf16 (round to nearest even), eval rows gathered, target scores
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_items_bf16_kernel(const float *__restrict__ I, int64_t n4, __nv_bfloat16 *out) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n4; t += (int64_t)gridDim.x * blockDim.x) {
        const float4 x = ldg4(I + 4 * t);
        __nv_bfloat162 lo = __floats2bfloat162_rn(x.x, x.y), hi = __floats2bfloat162_rn(x.z, x.w);
        uint2 o;
        o.x = *reinterpret_cast<uint32_t *>(&lo);
        o.y = *reinterpret_cast<uint32_t *>(&hi);
        reinterpret_cast<uint2 *>(out)[t] = o;
    }
}

// one warp per eval row: A[r] = bf16(U[user_r]); target[r] = sum_d bf16(U[u,d]) * bf16(I[pos,d]) (fp32 FMA chain)
__global__ void __launch_bounds__(256) pack_users_kernel(const float *__restrict__ U, const float *__restrict__ I,
                                                          const int64_t *user, const int64_t *pos, int64_t R,
                                                          int64_t n_users, int64_t n_items, int D, __nv_bfloat16 *A,
                                                          float *target, uint8_t *row_ok, WrWorkspace *ws) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < R; r += nwarps) {
        const int64_t u = user[r], it = pos[r];
        const bool ok = (uint64_t)u < (uint64_t)n_users && (uint64_t)it < (uint64_t)n_items;
        float s = 0.f;
        for (int d = lane; d < D; d += 32) {
            float a = 0.f, b = 0.f;
            if (ok) {
                a = __bfloat162float(__float2bfloat16_rn(U[u * D + d]));
                b = __bfloat162float(__float2bfloat16_rn(I[it * D + d]));
            }
            A[r * D + d] = __float2bfloat16_rn(a);
            s = fmaf(a, b, s);
        }
        s = warp_sum(s);
        if (lane == 0) {
            target[r] = s;
            row_ok[r] = ok ? 1 : 0;
            if (!ok) atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
        }
    }
}

// item-shard mode: the user rows arrive gathered ([R, D], one per eval row) and the target scores are an input
__global__ void __launch_bounds__(256) pack_rows_kernel(const float *__restrict__ Urows, const int64_t *user, int64_t R,
                                                         int64_t n_users, int D, __nv_bfloat16 *A, uint8_t *row_ok,
                                                         WrWorkspace *ws) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < R; r += nwarps) {
        const bool ok = (uint64_t)user[r] < (uint64_t)n_users;
        for (int d = lane; d < D; d += 32) A[r * D + d] = __float2bfloat16_rn(ok ? Urows[r * D + d] : 0.f);
        if (lane == 0) {
            row_ok[r] = ok ? 1 : 0;
            if (!ok) atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
        }
    }
}

// ---- precision 2: a = hi + lo (+ residual <= 2^-16 |a|), both bf16 ----
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16 &hi, __nv_bfloat16 &lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));      // the difference is exact in fp32
}

// one warp per item: B'[j] = [hi | lo | hi] (3 D bf16); bmax = max_j ||b_j||_2 (non-negative floats order like their bits)
__global__ void __launch_bounds__(256) pack_items_split_kernel(const float *__restrict__ I, int64_t n_items, int D,
                                                                __nv_bfloat16 *out, uint32_t *bmax_bits) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    float mx = 0.f;
    for (int64_t j = warp; j < n_items; j += nwarps) {
        float ss = 0.f;
        for (int d = lane; d < D; d += 32) {
            const float x = I[j * D + d];
            __nv_bfloat16 hi, lo;
            split_bf16(x, hi, lo);
            __nv_bfloat16 *o = out + j * 3 * D;
            o[d] = hi;
            o[D + d] = lo;
            o[2 * D + d] = hi;
            ss = fmaf(x, x, ss);
        }
        ss = warp_sum(ss);
        mx = fmaxf(mx, sqrtf(ss) * 1.000001f);              // rounding of the sum of squares: never under-estimate
    }
    if (lane == 0 && mx > 0.f) atomicMax(bmax_bits, __float_as_uint(mx));
}

// one warp per eval row: A'[r] = [hi | hi | lo] ([hi | lo] if a_hilo); target[r] = precision 0's FMA chain over the
// UNROUNDED fp32 rows; anorm[r] = ||a_r||_2.  rows_gathered != 0: U holds one row per eval row (item-shard mode) and
// target is an input.
__global__ void __launch_bounds__(256) pack_users_split_kernel(const float *__restrict__ U, const float *__restrict__ I,
                                                                const int64_t *user, const int64_t *pos, int64_t R,
                                                                int64_t n_users, int64_t n_items, int D, int rows_gathered,
                                                                int a_hilo, __nv_bfloat16 *A, float *target, float *anorm,
                                                                uint8_t *row_ok, WrWorkspace *ws) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < R; r += nwarps) {
        const int64_t u = user[r];
        const int64_t it = rows_gathered ? 0 : pos[r];
        const bool ok = (uint64_t)u < (uint64_t)n_users && (rows_gathered || (uint64_t)it < (uint64_t)n_items);
        const float *a = U + (rows_gathered ? r : u) * D;
        float ss = 0.f;
        for (int d = lane; d < D; d += 32) {
            const float x = ok ? a[d] : 0.f;
            __nv_bfloat16 hi, lo;
            split_bf16(x, hi, lo);
            __nv_bfloat16 *o = A + r * (a_hilo ? 2 : 3) * D;
            o[d] = hi;
            if (a_hilo) {
                o[D + d] = lo;
            } else {
                o[D + d] = hi;
                o[2 * D + d] = lo;
            }
            ss = fmaf(x, x, ss);
        }
        ss = warp_sum(ss);
        if (lane == 0) {
            anorm[r] = sqrtf(ss) * 1.000001f;
            row_ok[r] = ok ? 1 : 0;
            if (!ok) atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
            if (!rows_gathered) {
                float s = 0.f;                               // eval_kernels.cu: s = fmaf(a_d, b_d, s), d = 0 .. D-1
                if (ok) {
                    const float *b = I + it * D;
                    for (int d = 0; d < D; ++d) s = fmaf(a[d], b[d], s);
                }
                target[r] = s;
            }
        }
    }
}

// The pairs whose tensor-core score fell inside the band: precision 0's FMA chain decides them.
__global__ void __launch_bounds__(256) eval_recheck_kernel(const uint2 *__restrict__ cand, const unsigned long long *cnt,
                                                            unsigned long long cap, const float *__restrict__ U,
                                                            const int64_t *user, int rows_gathered,
                                                            const float *__restrict__ I, int D, const float *__restrict__ target,
                                                            int32_t *rank) {
    unsigned long long n = *cnt;
    if (n > cap) n = cap;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint2 e = cand[i];
        const int64_t r = e.x;
        const float *a = U + (rows_gathered ? r : user[r]) * D, *b = I + (int64_t)e.y * D;
        float s = 0.f;
        for (int d = 0; d < D; d += 4) {
            const float4 x = ldg4(a + d), y = ldg4(b + d);
            s = fmaf(x.x, y.x, s);
            s = fmaf(x.y, y.y, s);
            s = fmaf(x.z, y.z, s);
            s = fmaf(x.w, y.w, s);
        }
        if (s > target[r]) atomicAdd(rank + r, 1);
    }
}

// ordering of candidates: higher value first, lower id first among equal values
__device__ __forceinline__ bool top_worse(float v, int32_t id, float w, int32_t wid) {
    return v < w || (v == w && id > wid);
}

// Precision 2 with top-k, one warp per row: the row's candidates (a superset of precision 0's top k, see the drain warps)
// are re-scored with precision 0's FMA chain, one candidate per lane, and merged into a sorted list (lane = slot) by
// (value desc, id asc), as eval_rank_kernel does.  Slots left empty are written as (-inf, -1), as precision 0 writes them.
// A row whose segment overflowed gets topk_idx[r, 0] = -2 and WR_STATUS_TOPK_OVERFLOW: the caller reruns it.
__global__ void __launch_bounds__(256) eval_topk_select_kernel(const int32_t *__restrict__ seg,
                                                                const int32_t *__restrict__ seg_cnt, int64_t R,
                                                                const float *__restrict__ U, const int64_t *user,
                                                                int rows_gathered, const float *__restrict__ I, int D,
                                                                int k, int32_t *topk_idx, float *topk_val, uint32_t *status) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const uint32_t kmask = k >= 32 ? 0xffffffffu : ((1u << k) - 1u);
    for (int64_t r = warp; r < R; r += nwarps) {
        const int n = seg_cnt[r];
        if (n > TC_SEG_CAP) {
            if (lane < k) {
                topk_val[r * k + lane] = -INFINITY;
                topk_idx[r * k + lane] = lane == 0 ? -2 : -1;
            }
            if (lane == 0) atomicOr(status, WR_STATUS_TOPK_OVERFLOW);
            continue;
        }
        const float *a = U + (rows_gathered ? r : user[r]) * D;
        float tv = -INFINITY, tau = -INFINITY;          // slot value; empty slots are worse than any candidate
        int32_t ti = INT32_MAX, taui = INT32_MAX;
        for (int c0 = 0; c0 < n; c0 += 32) {
            const int c = c0 + lane;
            float s = -INFINITY;
            int32_t id = INT32_MAX;
            if (c < n) {
                id = seg[r * TC_SEG_CAP + c];
                const float *b = I + (int64_t)id * D;
                s = 0.f;                                 // eval_kernels.cu: s = fmaf(a_d, b_d, s), d = 0 .. D-1
                for (int d = 0; d < D; d += 4) {
                    const float4 x = ldg4(a + d), y = ldg4(b + d);
                    s = fmaf(x.x, y.x, s);
                    s = fmaf(x.y, y.y, s);
                    s = fmaf(x.z, y.z, s);
                    s = fmaf(x.w, y.w, s);
                }
            }
            uint32_t pend = __ballot_sync(0xffffffffu, c < n && top_worse(tau, taui, s, id));
            while (pend) {
                const int src = __ffs(pend) - 1;
                pend &= pend - 1;
                const float v = __shfl_sync(0xffffffffu, s, src);
                const int32_t vid = __shfl_sync(0xffffffffu, id, src);
                if (!top_worse(tau, taui, v, vid)) continue;
                const int ins = __popc(__ballot_sync(0xffffffffu, !top_worse(tv, ti, v, vid)) & kmask);
                const float up_v = __shfl_up_sync(0xffffffffu, tv, 1);
                const int32_t up_i = __shfl_up_sync(0xffffffffu, ti, 1);
                if (lane == ins) {
                    tv = v;
                    ti = vid;
                } else if (lane > ins) {
                    tv = up_v;
                    ti = up_i;
                }
                tau = __shfl_sync(0xffffffffu, tv, k - 1);
                taui = __shfl_sync(0xffffffffu, ti, k - 1);
            }
        }
        if (lane < k) {
            const bool empty = ti == INT32_MAX;
            topk_val[r * k + lane] = empty ? -INFINITY : tv;
            topk_idx[r * k + lane] = empty ? -1 : ti;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// the scoring kernel
// ---------------------------------------------------------------------------------------------------------
constexpr int TC_BM = 128, TC_BN = 256;
constexpr int TC_EPI_WARPS = 16;                       // 4 per TMEM lane quarter, 64 accumulator columns each
constexpr int TC_THREADS = (4 + TC_EPI_WARPS) * 32;

// K = contraction length in bf16 elements (D for precision 1, 3 D for precision 2).  A (128 x K) is loaded once per CTA;
// B travels through a ring of stages of SKB 64-element K blocks (32 KB each) of one 256-item tile: a whole tile per
// stage for precision 1 (one barrier round per tile: 5 % faster at D = 128 than block-wise staging) as long as two such
// stages fit, else half a tile (D = 256: two 64 KB stages beside the 64 KB of A); one K block per stage for precision 2,
// whose tiles (96 / 192 / 384 KB) would not fit twice.
// Precision 2 at D = 256: A' = [hi | hi | lo] would take 192 KB and leave no room for a ring, so only [hi | lo] (128 KB)
// is resident (A_HILO) and the MMAs of K blocks KB/3 .. 2 KB/3 - 1 read the hi blocks again; two 32 KB B stages fit.
__host__ __device__ constexpr bool exact_a_hilo(int D) { return D >= 256; }
// K blocks per B stage: the whole tile if two stages of it fit in room_kblocks, else the largest power-of-two share
__host__ __device__ constexpr int tc_stage_kblocks(int kb, int room_kblocks) {
    return kb > 1 && room_kblocks < 2 * kb ? tc_stage_kblocks(kb / 2, room_kblocks) : kb;
}
constexpr int TC_CAND_BUF = 64;                        // candidate entries buffered per epilogue warp (precision 2)
// top-k mode 2 (below): per-row rings in shared memory, drained by four extra warps
constexpr int TC_RING = 16;                             // ring entries per row
constexpr int TC_DRAIN_WARPS = 4;
constexpr int TC_THREADS_DRAIN = TC_THREADS + TC_DRAIN_WARPS * 32;
constexpr int TC_SMEM_DRAIN = TC_BM * TC_RING * 8 + TC_BM * 12 + 64;      // rings, head / tail / tau per row, counters
// MT = 128-row A tiles per CTA.  MT = 1 (default): 128 rows x 256-item tiles; MT = 2 (WR_TC_VARIANT=12): 256 rows x
// 128-item tiles -- the same 32,768 scores and the same 512 TMEM columns per tile, but every B byte that leaves L2 feeds
// twice the rows.  Built to test whether the 6 TB/s of L2 reads (the item table is streamed once per 128 rows) is what
// holds the kernel at 36 % tensor-pipe activity at D = 64: it is not -- 43.3 ms against 43.2 ms at D = 64, 60.2 against
// 59.6 at D = 128 (profiles/r02_eval_variants.txt).  ncu: 0.745 instructions issued per cycle per SM sub-partition, ALU
// pipe 65 % busy: the epilogue's ~4.5 issue slots per score (2 for the count, the rest mask / cursor / loop overhead per
// 32-column chunk) are the limiter at D = 64.  At D = 256 MT = 2 still fits (128 KB of A, two 32 KB half-tile stages).
// TOPK only matters for precision 2: its top-k instantiation takes the drain state out of the ring's room (D = 64: four
// stages instead of five; D = 128 / 256 keep three / two), the ranks-only configurations are untouched.  Precision 1
// reserves 19 KB for the drain state whether or not a call asks for lists.
template <int K, int EXACT, int MT, int TOPK = 0>
struct TcCfg {
    static constexpr int BM = TC_BM * MT;                  // rows per CTA
    static constexpr int BN = MT == 2 ? 128 : TC_BN;       // items per tile
    static constexpr int KB = K / 64;                      // 64-element (128 B) K blocks
    static constexpr bool A_HILO = EXACT && exact_a_hilo(K / 3);
    static constexpr int A_KB = A_HILO ? 2 * KB / 3 : KB;  // resident K blocks of A
    static constexpr int KBLOCK_BYTES = BN * 128;
    static constexpr int A_BYTES = BM * A_KB * 128;
    static constexpr int TAIL = 256 /*barriers*/ + 4 * TC_BM * 4 /*counts*/ + (EXACT ? TC_EPI_WARPS * TC_CAND_BUF * 8 : 0);
    static constexpr int ROOM = 227 * 1024 - 1024 - A_BYTES - TAIL - (MT == 1 && !EXACT ? 19 * 1024 : 0) /*top-k drain state*/
                                - (EXACT && TOPK == 2 ? TC_SMEM_DRAIN : 0);
    static constexpr int SKB = EXACT ? 1 : tc_stage_kblocks(KB, ROOM / KBLOCK_BYTES);      // K blocks per stage
    static constexpr int STAGE_BYTES = SKB * KBLOCK_BYTES;
    static constexpr int STAGES = ROOM / STAGE_BYTES > 6 ? 6 : ROOM / STAGE_BYTES;
    static_assert(STAGES >= 2, "the B ring needs two stages");
    static constexpr int SMEM = 1024 /*align slack*/ + A_BYTES + STAGES * STAGE_BYTES + TAIL;
};

// Top-k state of one epilogue thread (one row, one 64-column stripe of every tile), in local memory:
//   - the k best scores seen so far, UNSORTED, with the position of the worst of them; tau = its value.  A new
//     entry overwrites the worst one and the new worst is found by one pass of k independent loads (no dependent
//     shift chain: local memory is an L2 round trip away here, the shared memory being given to the operand ring);
//   - an unsorted buffer that scores beating tau are APPENDED to.
// The buffers of a warp are folded into the lists together ("compaction", warp-synchronous) when any lane's buffer
// could overflow on the next chunk, so the insertions of the 32 rows run side by side instead of one lane at a time.
// After the first tiles a score beats tau about k/m of the time (m = scores seen by the thread).
constexpr int TC_TOPBUF = 64;
struct TopState {
    float lv[TC_KMAX];
    int32_t li[TC_KMAX];
    float bv[TC_TOPBUF];
    int32_t bi[TC_TOPBUF];
};
__device__ __noinline__ void top_compact(TopState &t, int k, int &bcnt, float &tau, int &worst) {
    const int most = __reduce_max_sync(0xffffffffu, bcnt);
    for (int i = 0; i < most; ++i) {
        if (i < bcnt) {
            const float v = t.bv[i];
            if (v > tau) {                       // ids arrive ascending: a tie with the worst kept entry loses
                t.lv[worst] = v;
                t.li[worst] = t.bi[i];
                float w = t.lv[0];
                int32_t wid = t.li[0];
                int wp = 0;
                for (int j = 1; j < k; ++j) {
                    const float x = t.lv[j];
                    const int32_t xid = t.li[j];
                    if (top_worse(x, xid, w, wid)) {
                        w = x;
                        wid = xid;
                        wp = j;
                    }
                }
                worst = wp;
                tau = w;
            }
        }
    }
    bcnt = 0;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// Precision 2 with top-k: a score t_j can be in precision 0's top k only if t_j >= tau_final - 2 eps_r (DESIGN.md
// section 4.3); tau only grows, so the test against the current tau keeps a superset.  eps here is c_D ||a_r|| max ||b||,
// twice the bound on |t - s|; the 2.4e-7 |tau| term covers the rounding of the subtraction.  -inf stays -inf.
__device__ __forceinline__ float exact_topk_floor(float tau, float eps) {
    return tau - (2.f * eps + 2.4e-7f * fabsf(tau));
}

// Top-k mode 2: the epilogue warps only FILTER -- a score that reaches the row's current k-th best is pushed into the
// row's ring in shared memory -- and four extra warps (one thread per row) drain the rings into per-row k-best
// lists and publish the new threshold.  The epilogue never sorts, never compacts and never waits for another
// epilogue warp's bookkeeping, and the threshold is per ROW (all 256 columns of a tile), not per 64-column stripe.

__device__ __forceinline__ uint32_t lds_vol_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_vol_u32(uint32_t a, uint32_t v) {
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

struct TopRings {
    float *v;                 // [TC_BM][TC_RING]
    int32_t *id;              // [TC_BM][TC_RING]   -1 = empty
    uint32_t *head, *tail;    // [TC_BM] monotonically increasing slot counters
    float *tau;               // [TC_BM] value of the row's k-th best so far (-inf until the list is full)
    int *epi_done;            // epilogue warps that have finished
};
__device__ __forceinline__ void ring_push(const TopRings &rg, int row, float x, int32_t id) {
    const uint32_t slot = atomicAdd(rg.head + row, 1u);
    const int o = row * TC_RING + (int)(slot & (TC_RING - 1));
    // The payload is written inside the iteration that finds room: a lane with room must never wait for the lanes
    // of its warp whose rings are full (their drainers may be waiting for THIS lane's payload).
    bool pending = true;
    while (pending) {
        if ((int32_t)(slot - *reinterpret_cast<volatile uint32_t *>(rg.tail + row)) < TC_RING) {
            *reinterpret_cast<volatile float *>(rg.v + o) = x;
            __threadfence_block();
            *reinterpret_cast<volatile int32_t *>(rg.id + o) = id;
            pending = false;
        }
    }
}

// LONG (precision 2 with TOPK = 2 only, wr_eval_rank_topk_long): 1 = bound pass -- the drain warps keep the k'-best list
// of this CTA's item range (blockIdx.y) and write its k'-th best t, no segment; 2 = collect pass -- the row's threshold is
// fixed at long_bound of its range bounds and every item the epilogue pushes (t >= that bound - 2 eps_r) goes to its
// segment.
template <int K, int VARIANT, int TOPK, int EXACT, int MT, int LONG = 0>
__global__ void __launch_bounds__(TOPK == 2 ? TC_THREADS_DRAIN : TC_THREADS, 1)
eval_tc_rank_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, TcParams p) {
    using C = TcCfg<K, EXACT, MT, TOPK>;
    static_assert(MT == 1 || TOPK == 0, "the top-k lists are laid out for 128 rows per CTA");
    static_assert(!EXACT || TOPK != 1, "precision 2 builds its lists with the drain warps");
    static_assert(LONG == 0 || (EXACT && TOPK == 2), "long lists are a precision-2 drain-warp mode");
    static_assert(TOPK != 1 || C::STAGES * C::STAGE_BYTES >= TC_BM * 4 * TC_KMAX * 8, "stripe lists fit in the B ring");
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = smem;
    uint8_t *sB = smem + C::A_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sB + C::STAGES * C::STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + C::STAGES, *a_full = bars + 2 * C::STAGES;
    uint64_t *tm_full = a_full + 1, *tm_empty = tm_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tm_empty + 2);
    int *cnt_s = reinterpret_cast<int *>(reinterpret_cast<uint8_t *>(bars) + 256);   // [4][128]
    uint2 *cand_s = reinterpret_cast<uint2 *>(cnt_s + 4 * TC_BM);                     // [TC_EPI_WARPS][TC_CAND_BUF], precision 2
    TopRings rg;
    rg.v = reinterpret_cast<float *>(cand_s + (EXACT ? TC_EPI_WARPS * TC_CAND_BUF : 0));
    rg.id = reinterpret_cast<int32_t *>(rg.v + TC_BM * TC_RING);
    rg.head = reinterpret_cast<uint32_t *>(rg.id + TC_BM * TC_RING);
    rg.tail = rg.head + TC_BM;
    rg.tau = reinterpret_cast<float *>(rg.tail + TC_BM);
    rg.epi_done = reinterpret_cast<int *>(rg.tau + TC_BM);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row0 = (int64_t)blockIdx.x * C::BM;
    const int t0 = blockIdx.y * p.tiles_per_split;
    const int t1 = min(p.n_tiles, t0 + p.tiles_per_split);

    if (threadIdx.x == 0) {
        for (int s = 0; s < C::STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(a_full, 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tm_full[s], 1);
            mbar_init(&tm_empty[s], TC_EPI_WARPS * 32);   // every epilogue thread arrives
        }
        fence_barrier_init();
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (TOPK == 2 && threadIdx.x >= TC_THREADS) {
        const int r = threadIdx.x - TC_THREADS;
        for (int i = 0; i < TC_RING; ++i) rg.id[r * TC_RING + i] = -1;
        rg.head[r] = 0;
        rg.tail[r] = 0;
        rg.tau[r] = LONG == 2 && row0 + r < p.R ? long_bound(p.bound + (row0 + r) * WR_LONG_RANGES, p.n_bounds, p.bound_need)
                                                : -INFINITY;
        if (r == 0) *rg.epi_done = 0;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ---------------- TMA producer ----------------
            mbar_expect_tx(a_full, C::A_BYTES);
#pragma unroll
            for (int kb = 0; kb < C::A_KB; ++kb)
                for (int mh = 0; mh < MT; ++mh)
                    tma_load_2d(&tmA, a_full, sA + (mh * C::A_KB + kb) * (TC_BM * 128), kb * 64, (int)row0 + mh * TC_BM);
            int it = 0;
            for (int t = t0; t < t1; ++t) {
#pragma unroll 1
                for (int kb0 = 0; kb0 < C::KB; kb0 += C::SKB, ++it) {
                    const int stage = it % C::STAGES;
                    const uint32_t ph = (it / C::STAGES) & 1;
                    mbar_wait(&empty[stage], ph ^ 1);
                    mbar_expect_tx(&full[stage], C::STAGE_BYTES);
#pragma unroll
                    for (int kb = 0; kb < C::SKB; ++kb)
                        tma_load_2d(&tmB, &full[stage], sB + stage * C::STAGE_BYTES + kb * C::KBLOCK_BYTES, (kb0 + kb) * 64,
                                    t * C::BN);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ---------------- MMA issuer ----------------
            constexpr uint32_t idesc = umma_idesc_bf16(TC_BM, C::BN);
            mbar_wait(a_full, 0);
            tc_fence_after();
            int it = 0;
            for (int t = t0, ti = 0; t < t1; ++t, ++ti) {
                const int acc = ti & 1;
                const uint32_t aph = (ti >> 1) & 1;
                mbar_wait(&tm_empty[acc], aph ^ 1);          // epilogue has drained this accumulator
                const uint32_t d_tmem = tmem_base + acc * MT * C::BN;      // MT accumulators of BN columns per buffer
#pragma unroll 1
                for (int kb0 = 0; kb0 < C::KB; kb0 += C::SKB, ++it) {
                    const int stage = it % C::STAGES;
                    const uint32_t ph = (it / C::STAGES) & 1;
                    mbar_wait(&full[stage], ph);             // TMA has landed this stage
                    tc_fence_after();
#pragma unroll
                    for (int kb = 0; kb < C::SKB; ++kb) {
                        const uint64_t b0 = umma_desc_sw128(sB + stage * C::STAGE_BYTES + kb * C::KBLOCK_BYTES);
                        // A_HILO: K blocks of the middle third (B's lo) pair with A's hi blocks, the last third with lo
                        const int akb = C::A_HILO && kb0 + kb >= C::KB / 3 ? kb0 + kb - C::KB / 3 : kb0 + kb;
#pragma unroll
                        for (int mh = 0; mh < MT; ++mh) {   // the two row halves share the B tile
                            const uint64_t a0 = umma_desc_sw128(sA + (mh * C::A_KB + akb) * (TC_BM * 128));
#pragma unroll
                            for (int k = 0; k < 4; ++k)     // K = 16 bf16 = 32 B per instruction: +2 in the >>4 address field
                                umma_bf16(d_tmem + mh * C::BN, a0 + 2 * k, b0 + 2 * k, idesc, (kb0 | kb | k) != 0);
                        }
                    }
                    umma_commit(&empty[stage]);              // frees the smem stage when the MMAs retire
                }
                umma_commit(&tm_full[acc]);                  // accumulator ready for the epilogue
            }
        }
    } else if (warp >= 4 && warp < 4 + TC_EPI_WARPS) {
        // ---------------- epilogue: 16 warps, TMEM lane quarter = warp % 4, column group = (warp - 4) / 4 ----------------
        const int quarter = warp & 3, widx = (warp - 4) >> 2;
        const int mh = MT == 2 ? widx >> 1 : 0;             // which 128-row half this warp reads
        const int grp = MT == 2 ? (widx & 1) : widx;        // which 64-column stripe of the tile
        const int rl = mh * TC_BM + quarter * 32 + lane;
        const int64_t r = row0 + rl;
        bool live = false;
        float st = 0.f;
        int64_t cur = 0, hend = 0;
        int32_t posj = -1;
        int32_t next_h = INT32_MAX;                       // next history item of this row, cached in a register
        const int32_t n_items = (int32_t)p.n_items;
        if (r < p.R && p.row_ok[r]) {
            live = true;
            st = p.target[r];
            const int64_t u = p.user[r];
            posj = (int32_t)p.pos[r];
            cur = p.hist_ptr[u];
            hend = p.hist_ptr[u + 1];
            const int32_t first = (int32_t)min((int64_t)t0 * C::BN, (int64_t)INT32_MAX);
            int64_t lo = cur, hi = hend;
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (p.hist_idx[mid] < first) lo = mid + 1; else hi = mid;
            }
            cur = lo;
            if (cur < hend) next_h = __ldg(p.hist_idx + cur);
        }
        int cnt = 0;
        // precision 2: scores above st_hi certainly beat the target in precision 0's arithmetic, scores below st_lo
        // certainly do not; the band between them goes to the candidate list
        float st_hi = st, st_lo = st;
        int ccount = 0;                                        // candidates buffered by this warp (warp-uniform)
        uint2 *cbuf = cand_s + (warp - 4) * TC_CAND_BUF;
        float eps_top = 0.f;                                   // precision-2 top-k: |t - s| <= eps_top / 2 for every item
        if (EXACT && live) {
            const float eps = p.band_c * p.anorm[r] * p.bmax[0] + 2.4e-7f * fabsf(st);
            st_hi = st + eps;
            st_lo = st - eps;
            if (TOPK == 2) eps_top = p.band_c * p.anorm[r] * p.bmax[0];
        }
        TopState top;
        const int top_trigger = p.top_trigger;      // fold the buffers once any lane holds more than this many
        float tau = -INFINITY;
        int bcnt = 0, worst = 0;
        if (TOPK == 1) {
            for (int i = 0; i < p.k; ++i) {
                top.lv[i] = -INFINITY;
                top.li[i] = INT32_MAX - i;      // empty slots: worse than anything, distinct, evicted first
            }
        }
        for (int t = t0, it = 0; t < t1; ++t, ++it) {
            const int acc = it & 1;
            const uint32_t aph = (it >> 1) & 1;
            mbar_wait(&tm_full[acc], aph);
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < 2; ++c) {
                const int col0 = grp * 64 + c * 32;
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((acc * MT + mh) * C::BN + col0), v);
                const int32_t j0 = t * C::BN + col0;
                // columns of this chunk that must not count: history, past the table, the target itself
                uint32_t m = 0, m_top = 0;      // m_top: not a candidate (history, past the table); the target is one
                if (!live) {
                    m = m_top = 0xffffffffu;
                } else {
                    while (next_h < j0 + 32) {
                        if (next_h >= j0) m |= 1u << (next_h - j0);
                        ++cur;
                        next_h = cur < hend ? __ldg(p.hist_idx + cur) : INT32_MAX;
                    }
                    if (j0 + 32 > n_items) m |= j0 >= n_items ? 0xffffffffu : (0xffffffffu << (n_items - j0));
                    m_top = m;
                    const uint32_t pj = (uint32_t)(posj - j0);
                    if (pj < 32u) m |= 1u << pj;
                }
                tmem_ld_wait();
                if (TOPK == 2) {
                    if (m_top != 0) {       // history / table-end columns can never be candidates (the compiler turns
#pragma unroll                              // this into 32 selects: cheaper than a divergent branch per chunk)
                        for (int i = 0; i < 32; ++i)
                            if ((m_top >> i) & 1u) v[i] = 0xff800000u;      // -inf; these columns are in m as well
                    }
                    // the row's threshold as the drain warps last published it (stale = lower = still correct).
                    // ">=" lets ties through: the drainer decides them by item id.  Precision 2 lowers it by the
                    // band (tau - 2 eps_r, rounded down): such scores may still be in precision 0's top k
                    const float tau_pub = *reinterpret_cast<volatile float *>(rg.tau + rl);
                    const float tau_row = EXACT ? exact_topk_floor(tau_pub, eps_top) : tau_pub;
#pragma unroll
                    for (int g8 = 0; g8 < 32; g8 += 8) {
                        float mx = fmax3(__uint_as_float(v[g8]), __uint_as_float(v[g8 + 1]), __uint_as_float(v[g8 + 2]));
                        mx = fmax3(mx, __uint_as_float(v[g8 + 3]), __uint_as_float(v[g8 + 4]));
                        mx = fmax3(mx, __uint_as_float(v[g8 + 5]), __uint_as_float(v[g8 + 6]));
                        mx = fmaxf(mx, __uint_as_float(v[g8 + 7]));
                        if (mx >= tau_row && mx > -INFINITY) {
#pragma unroll
                            for (int i = g8; i < g8 + 8; ++i) {
                                const float x = __uint_as_float(v[i]);
                                if (x >= tau_row && x > -INFINITY) ring_push(rg, rl, x, j0 + i);
                            }
                        }
                    }
                }
                if (TOPK == 1) {
                    if (m_top != 0) {       // rare: history / table-end columns can never be candidates
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if ((m_top >> i) & 1u) v[i] = 0xff800000u;      // -inf; these columns are in m as well
                    }
                    // half an instruction per score (3-input max) finds out whether a group of 8 columns holds a
                    // candidate; only such a group (rare once tau has settled) pays for 8 predicated appends
#pragma unroll
                    for (int g8 = 0; g8 < 32; g8 += 8) {
                        float mx = fmax3(__uint_as_float(v[g8]), __uint_as_float(v[g8 + 1]), __uint_as_float(v[g8 + 2]));
                        mx = fmax3(mx, __uint_as_float(v[g8 + 3]), __uint_as_float(v[g8 + 4]));
                        mx = fmax3(mx, __uint_as_float(v[g8 + 5]), __uint_as_float(v[g8 + 6]));
                        mx = fmaxf(mx, __uint_as_float(v[g8 + 7]));
                        if (mx > tau) {
#pragma unroll
                            for (int i = g8; i < g8 + 8; ++i) {
                                const float x = __uint_as_float(v[i]);
                                if (x > tau) {
                                    top.bv[bcnt] = x;
                                    top.bi[bcnt] = j0 + i;
                                    ++bcnt;
                                }
                            }
                        }
                    }
                    if (__any_sync(0xffffffffu, bcnt > top_trigger)) top_compact(top, p.k, bcnt, tau, worst);
                }
                if (EXACT) {
                    uint32_t cm = 0;                            // columns of this chunk inside the band
                    bool bits = m != 0;
                    if (!bits) {
                        float h0 = 0.f, h1 = 0.f, l0 = 0.f, l1 = 0.f;
#define WR_CNT2(hi_, lo_, i_)                                                                                 \
    asm("{\n\t.reg .pred q;\n\tsetp.gt.f32 q, %2, %3;\n\t@q add.f32 %0, %0, 0f3F800000;\n\t"                  \
        "setp.ge.f32 q, %2, %4;\n\t@q add.f32 %1, %1, 0f3F800000;\n\t}"                                      \
        : "+f"(hi_), "+f"(lo_)                                                                                \
        : "f"(__uint_as_float(v[i_])), "f"(st_hi), "f"(st_lo))
#pragma unroll
                        for (int i = 0; i < 32; i += 2) {
                            WR_CNT2(h0, l0, i);
                            WR_CNT2(h1, l1, i + 1);
                        }
#undef WR_CNT2
                        const float hi_n = h0 + h1;
                        cnt += (int)hi_n;
                        bits = (l0 + l1) != hi_n;               // somebody is inside the band: find out who
                        if (bits) cnt -= (int)hi_n;
                    }
                    if (bits) {
                        uint32_t gt = 0, ge = 0;
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            const float x = __uint_as_float(v[i]);
                            gt |= (x > st_hi ? 1u : 0u) << i;
                            ge |= (x >= st_lo ? 1u : 0u) << i;
                        }
                        cnt += __popc(gt & ~m);
                        cm = ge & ~gt & ~m;
                    }
                    if (__any_sync(0xffffffffu, cm != 0)) {
                        const int nc = __popc(cm);
                        int incl = nc;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const int y = __shfl_up_sync(0xffffffffu, incl, o);
                            if (lane >= o) incl += y;
                        }
                        const int total = __shfl_sync(0xffffffffu, incl, 31);
                        int at = incl - nc;
                        if (ccount + total > TC_CAND_BUF && ccount > 0) {        // make room: buffer -> global list
                            unsigned long long base = 0;
                            if (lane == 0) base = atomicAdd(p.cand_cnt, (unsigned long long)ccount);
                            base = __shfl_sync(0xffffffffu, base, 0);
                            __syncwarp();
                            for (int i = lane; i < ccount; i += 32) {
                                if (base + i < p.cand_cap) p.cand[base + i] = cbuf[i];
                                else atomicOr(p.status, WR_STATUS_EVAL_OVERFLOW);
                            }
                            __syncwarp();
                            ccount = 0;
                        }
                        if (total > TC_CAND_BUF) {                               // a degenerate chunk: straight to the list
                            unsigned long long base = 0;
                            if (lane == 0) base = atomicAdd(p.cand_cnt, (unsigned long long)total);
                            base = __shfl_sync(0xffffffffu, base, 0);
                            while (cm) {
                                const int i = __ffs(cm) - 1;
                                cm &= cm - 1;
                                if (base + at < p.cand_cap) p.cand[base + at] = make_uint2((uint32_t)r, (uint32_t)(j0 + i));
                                else atomicOr(p.status, WR_STATUS_EVAL_OVERFLOW);
                                ++at;
                            }
                        } else {
                            while (cm) {
                                const int i = __ffs(cm) - 1;
                                cm &= cm - 1;
                                cbuf[ccount + at] = make_uint2((uint32_t)r, (uint32_t)(j0 + i));
                                ++at;
                            }
                            ccount += total;
                        }
                    }
                } else if (m == 0) {
                    // fast path, 2 instructions per score.  VARIANT 0: FSETP + predicated integer add (both ALU pipe);
                    // 1: FSETP (ALU) + predicated FADD (FMA pipe); 2: FFMA.SAT + FADD (FMA pipe only):
                    // sat(v*2^100 - st*2^100) is exactly [v > st]; 3: even columns as 1, odd columns as 2.
                    if (VARIANT == 0) {
                        int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#define WR_CNT(acc_, i_)                                                                                      \
    asm("{\n\t.reg .pred q;\n\tsetp.gt.f32 q, %1, %2;\n\t@q add.s32 %0, %0, 1;\n\t}"                          \
        : "+r"(acc_)                                                                                          \
        : "f"(__uint_as_float(v[i_])), "f"(st))
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            WR_CNT(c0, i);
                            WR_CNT(c1, i + 1);
                            WR_CNT(c2, i + 2);
                            WR_CNT(c3, i + 3);
                        }
#undef WR_CNT
                        cnt += (c0 + c1) + (c2 + c3);
                    } else {
                        float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f;
                        const float big = 1.2676506e30f;                 // 2^100
                        const float nst = -st * big;
#define WR_CNTP(acc_, i_)                                                                                     \
    asm("{\n\t.reg .pred q;\n\tsetp.gt.f32 q, %1, %2;\n\t@q add.f32 %0, %0, 0f3F800000;\n\t}"                 \
        : "+f"(acc_)                                                                                          \
        : "f"(__uint_as_float(v[i_])), "f"(st))
#define WR_CNTF(acc_, i_)                                                                                     \
    {                                                                                                         \
        float t_;                                                                                             \
        asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(t_) : "f"(__uint_as_float(v[i_])), "f"(big), "f"(nst));  \
        acc_ += t_;                                                                                           \
    }
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            if (VARIANT == 1) { WR_CNTP(f0, i); WR_CNTP(f1, i + 1); WR_CNTP(f2, i + 2); WR_CNTP(f3, i + 3); }
                            if (VARIANT == 2) { WR_CNTF(f0, i); WR_CNTF(f1, i + 1); WR_CNTF(f2, i + 2); WR_CNTF(f3, i + 3); }
                            if (VARIANT == 3) { WR_CNTP(f0, i); WR_CNTF(f1, i + 1); WR_CNTP(f2, i + 2); WR_CNTF(f3, i + 3); }
                        }
#undef WR_CNTP
#undef WR_CNTF
                        cnt += (int)((f0 + f1) + (f2 + f3));
                    }
                } else {
                    uint32_t gt = 0;
#pragma unroll
                    for (int i = 0; i < 32; ++i) gt |= (__uint_as_float(v[i]) > st ? 1u : 0u) << i;
                    cnt += __popc(gt & ~m);
                }
                if (p.scores && r < p.R) {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (j0 + i < n_items) p.scores[r * p.n_items + j0 + i] = __uint_as_float(v[i]);
                }
            }
            tc_fence_before();
            mbar_arrive(&tm_empty[acc]);
        }
        if (EXACT && ccount > 0) {                              // what is left in this warp's candidate buffer
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(p.cand_cnt, (unsigned long long)ccount);
            base = __shfl_sync(0xffffffffu, base, 0);
            __syncwarp();
            for (int i = lane; i < ccount; i += 32) {
                if (base + i < p.cand_cap) p.cand[base + i] = cbuf[i];
                else atomicOr(p.status, WR_STATUS_EVAL_OVERFLOW);
            }
        }
        // the four stripe lists of a row meet in the (now idle) B-stage shared memory: [row][stripe][k]
        float *lv = reinterpret_cast<float *>(sB);
        int32_t *li = reinterpret_cast<int32_t *>(sB + TC_BM * 4 * TC_KMAX * 4);
        if (TOPK == 1) {
            top_compact(top, p.k, bcnt, tau, worst);
            for (int i = 0; i < p.k; ++i) {
                lv[(rl * 4 + grp) * TC_KMAX + i] = top.lv[i];
                li[(rl * 4 + grp) * TC_KMAX + i] = top.li[i];
            }
        }
        if (TOPK == 2) {                    // every push of this warp is visible before the drain warps see "done"
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                atomicAdd(rg.epi_done, 1);
            }
        }
        cnt_s[grp * C::BM + rl] = cnt;
        asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_WARPS * 32) : "memory");      // the epilogue warps only
        if (grp == 0 && r < p.R) {
            const int total = MT == 2 ? cnt_s[rl] + cnt_s[C::BM + rl]
                                      : cnt_s[rl] + cnt_s[TC_BM + rl] + cnt_s[2 * TC_BM + rl] + cnt_s[3 * TC_BM + rl];
            if (p.splits == 1) p.rank[r] = 1 + total;
            else atomicAdd(&p.rank[r], total);
            if (TOPK == 1) {
                // the row's 4k candidates (unsorted) -> its k best in order: k selection passes, taken slots marked
                const int n = 4 * TC_KMAX;
                for (int s = 0; s < p.k; ++s) {
                    int best = -1;
                    float bv = 0.f;
                    int32_t bi = 0;
                    for (int o = 0; o < n; ++o) {
                        if ((o & (TC_KMAX - 1)) >= p.k) continue;
                        const int32_t id = li[rl * n + o];
                        if (id < 0 || id >= INT32_MAX - TC_KMAX) continue;      // taken / empty
                        const float x = lv[rl * n + o];
                        if (best < 0 || top_worse(bv, bi, x, id)) {
                            best = o;
                            bv = x;
                            bi = id;
                        }
                    }
                    if (best >= 0) li[rl * n + best] = -1;
                    p.topk_val[r * p.k + s] = best >= 0 ? bv : -INFINITY;
                    p.topk_idx[r * p.k + s] = best >= 0 ? bi : -1;
                }
            }
        }
    }
    if (TOPK == 2 && warp >= 4 + TC_EPI_WARPS) {
        // ---------------- drain warps: thread r owns row r's ring and its k-best list ----------------
        const int r = threadIdx.x - TC_THREADS;
        const int k = p.k;
        float lv[TC_KMAX];
        int32_t li[TC_KMAX];
        for (int i = 0; i < k; ++i) {
            lv[i] = -INFINITY;
            li[i] = INT32_MAX - i;                      // empty slots: worse than anything, distinct
        }
        float w = -INFINITY;                            // the worst kept entry: value, id, position
        int32_t wid = INT32_MAX;
        int wp = 0;
        uint32_t tail = 0;
        // precision 2: the k-best list above is over the tensor-core scores; what is kept is the row's candidate
        // segment -- every entry of the list and every score within the band of its k-th best on arrival
        const int64_t row = row0 + r;
        float e = 0.f;
        constexpr int SEG_CAP = LONG ? WR_LONG_SEG_CAP : TC_SEG_CAP;
        int nseg = 0;
        int32_t *segr = nullptr;
        if (EXACT && row < p.R) {
            e = p.band_c * p.anorm[row] * p.bmax[0];
            if (LONG != 1) segr = p.seg + row * SEG_CAP;
        }
        volatile uint32_t *vhead = rg.head + r;
        volatile int32_t *vid = rg.id + r * TC_RING;
        volatile float *vv = rg.v + r * TC_RING;
        while (true) {
            const bool finishing = *reinterpret_cast<volatile int *>(rg.epi_done) == TC_EPI_WARPS;
            const uint32_t head = *vhead;               // read AFTER the completion count: if that was final, so is this
            if (tail == head) {
                if (finishing) break;
                __nanosleep(100);
                continue;
            }
            while (tail != head) {
                const int o = (int)(tail & (TC_RING - 1));
                int32_t id;
                while ((id = vid[o]) == -1) {}          // slot claimed, payload still on its way
                __threadfence_block();
                const float x = vv[o];
                vid[o] = -1;
                __threadfence_block();
                ++tail;
                *reinterpret_cast<volatile uint32_t *>(rg.tail + r) = tail;
                bool keep = LONG == 2;                  // collect pass: every push is a candidate, tau stays put
                if (LONG != 2 && top_worse(w, wid, x, id)) {    // beats the worst kept entry (ties: the lower id wins)
                    keep = true;
                    lv[wp] = x;
                    li[wp] = id;
                    w = lv[0];
                    wid = li[0];
                    wp = 0;
                    for (int j = 1; j < k; ++j) {
                        if (top_worse(lv[j], li[j], w, wid)) {
                            w = lv[j];
                            wid = li[j];
                            wp = j;
                        }
                    }
                    *reinterpret_cast<volatile float *>(rg.tau + r) = w;
                } else if (LONG == 0 && EXACT && e > 0.f && x >= exact_topk_floor(w, e)) {
                    keep = true;                        // below the list but within 2 eps_r of its k-th best
                }
                if (EXACT && LONG != 1 && keep) {
                    if (nseg < SEG_CAP) segr[nseg] = id;
                    ++nseg;
                }
            }
        }
        if (LONG == 1) {
            if (row < p.R) p.bound[row * WR_LONG_RANGES + blockIdx.y] = w;     // -inf: fewer than k' items in range
        } else if (EXACT) {
            if (row < p.R) p.seg_cnt[row] = nseg;
        } else if (row < p.R) {
            for (int s = 0; s < k; ++s) {               // k selection passes: best first
                int best = -1;
                for (int j = 0; j < k; ++j) {
                    if (li[j] < 0 || li[j] >= INT32_MAX - TC_KMAX) continue;        // taken / empty
                    if (best < 0 || top_worse(lv[best], li[best], lv[j], li[j])) best = j;
                }
                p.topk_val[row * k + s] = best >= 0 ? lv[best] : -INFINITY;
                p.topk_idx[row * k + s] = best >= 0 ? li[best] : -1;
                if (best >= 0) li[best] = -1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
    }
}

__global__ void fill_rank_kernel(int32_t *x, int64_t n, int32_t v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] = v;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_map(CUtensorMap *map, const void *base, int64_t rows, int D /* bf16 elements per row */, int box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q);
        if (e != cudaSuccess) return (int)e;
        if (!sym || q != cudaDriverEntryPointSuccess) return (int)cudaErrorNotSupported;
        fn = (EncodeTiledFn)sym;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)D, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)D * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

template <int K, int VARIANT, int TOPK, int EXACT, int MT, int LONG = 0>
static int launch_tc_v(const CUtensorMap &ma, const CUtensorMap &mb, TcParams &p, int row_tiles, cudaStream_t st) {
    constexpr int smem = TcCfg<K, EXACT, MT, TOPK>::SMEM + (TOPK == 2 ? TC_SMEM_DRAIN : 0);
    constexpr int threads = TOPK == 2 ? TC_THREADS_DRAIN : TC_THREADS;
    static_assert(smem <= 227 * 1024, "shared memory budget");
    cudaError_t e = cudaFuncSetAttribute(eval_tc_rank_kernel<K, VARIANT, TOPK, EXACT, MT, LONG>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    eval_tc_rank_kernel<K, VARIANT, TOPK, EXACT, MT, LONG><<<dim3(row_tiles, p.splits), threads, smem, st>>>(ma, mb, p);
    return (int)cudaGetLastError();
}

static int tc_variant() {
    static int variant = -1;
    if (variant < 0) {
        const char *e = getenv("WR_TC_VARIANT");        // tuning knob: the epilogue's counting form; 12 = 256 rows per CTA
        variant = e ? atoi(e) : 1;
    }
    return variant;
}

template <int D>
static int launch_tc(const CUtensorMap &ma, const CUtensorMap &mb, TcParams &p, int row_tiles, cudaStream_t st) {
    const int variant = tc_variant();
    if (p.topk_idx) {
        static int mode = -1;
        if (mode < 0) {
            const char *e = getenv("WR_TC_TOPK_MODE");      // 1: per-thread lists in the epilogue; 2: drain warps
            mode = e ? atoi(e) : 2;
        }
        return mode == 1 ? launch_tc_v<D, 1, 1, 0, 1>(ma, mb, p, row_tiles, st) : launch_tc_v<D, 1, 2, 0, 1>(ma, mb, p, row_tiles, st);
    }
    switch (variant) {
        case 1: return launch_tc_v<D, 1, 0, 0, 1>(ma, mb, p, row_tiles, st);
        case 2: return launch_tc_v<D, 2, 0, 0, 1>(ma, mb, p, row_tiles, st);
        case 3: return launch_tc_v<D, 3, 0, 0, 1>(ma, mb, p, row_tiles, st);
        case 12: return launch_tc_v<D, 1, 0, 0, 2>(ma, mb, p, row_tiles, st);      // 256 rows per CTA (see TcCfg)
        default: return launch_tc_v<D, 0, 0, 0, 1>(ma, mb, p, row_tiles, st);
    }
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bf16 columns of the packed user rows: D (precision 1), 3 D = [hi | hi | lo] or, at D = 256, 2 D = [hi | lo] (precision 2)
static inline int tc_a_cols(int D, bool exact) { return !exact ? D : exact_a_hilo(D) ? 2 * D : 3 * D; }

// c_D of the precision-2 band: twice the worst-case sum of the dropped lo.lo term (3.1 2^-16), the fp32 accumulation of
// 3 D products (3 D 2^-23) and precision 0's own FMA chain (D 2^-24), rounded up -- DESIGN.md section 4.3
static inline float exact_band_c(int D) {
    switch (D) {
        case 64: return 1.5e-4f;        // 2 x 7.40e-5
        case 128: return 2.0e-4f;       // 2 x 1.007e-4
        default: return 3.1e-4f;        // D = 256: 2 x 1.542e-4
    }
}

}  // namespace wr

using namespace wr;

// precision 2: rows are evaluated in blocks so that the candidate list (one (row, item) pair per score inside the band,
// ~0.1 % of the pairs; sized for 0.8 %) stays below 1 GB
static void exact_blocking(int64_t R, int64_t n_items, int64_t *rows_per_block, unsigned long long *cand_cap) {
    int64_t rb = (int64_t)(16e9 / (double)n_items);
    rb = rb / (2 * TC_BM) * (2 * TC_BM);
    if (rb < 2 * TC_BM) rb = 2 * TC_BM;
    if (rb > R) rb = (R + 2 * TC_BM - 1) / (2 * TC_BM) * (2 * TC_BM);
    unsigned long long cap = (unsigned long long)((double)rb * (double)n_items / 128.0);
    if (cap < (1ull << 20)) cap = 1ull << 20;
    if (cap > (1ull << 27)) cap = 1ull << 27;
    *rows_per_block = rb;
    *cand_cap = cap;
}

// precision 2 with top-k: the same blocks, at most 262,144 rows so that the candidate segments (4 KB per row) stay <= 1 GB
static void exact_blocking_topk(int64_t R, int64_t n_items, int k, int64_t *rows_per_block, unsigned long long *cand_cap) {
    exact_blocking(R, n_items, rows_per_block, cand_cap);
    const int64_t most = ((int64_t)1 << 30) / ((int64_t)TC_SEG_CAP * 4);
    if (k > 0 && *rows_per_block > most) *rows_per_block = most;
}

// long lists: the same blocks, at most WR_LONG_BLOCK_ROWS rows so that the segments (16 KB per row) stay <= 1 GB
static int64_t exact_blocking_long(int64_t R, int64_t n_items) {
    int64_t rb;
    unsigned long long cap;
    exact_blocking(R, n_items, &rb, &cap);
    return rb < WR_LONG_BLOCK_ROWS ? rb : WR_LONG_BLOCK_ROWS;
}

extern "C" size_t wr_eval_scratch_bytes(int64_t R, int64_t n_items, int D, int precision) {
    if ((precision != 1 && precision != 2) || R <= 0 || n_items <= 0 || D <= 0) return 0;
    const size_t k = precision == 2 ? 3 : 1;
    size_t n = align_up((size_t)R * tc_a_cols(D, precision == 2) * 2, 1024) + align_up((size_t)n_items * D * 2 * k, 1024) +
               align_up((size_t)R, 1024) + 1024;
    if (precision == 2) {
        int64_t rb;
        unsigned long long cap;
        exact_blocking(R, n_items, &rb, &cap);
        n += align_up((size_t)R * 4, 1024) + 1024 + (size_t)cap * 8;
    }
    return n;
}

extern "C" size_t wr_eval_scratch_bytes_topk(int64_t R, int64_t n_items, int D, int precision, int k) {
    const size_t n = wr_eval_scratch_bytes(R, n_items, D, precision);
    if (precision != 2 || k <= 0 || n == 0) return n;
    int64_t rb;
    unsigned long long cap;
    exact_blocking_topk(R, n_items, k, &rb, &cap);
    return n + 1024 + align_up((size_t)rb * 4, 1024) + (size_t)rb * TC_SEG_CAP * 4;      // counts, then segments
}

// A long call (wr_eval_rank_topk_long) needs a 1,024-byte header; precision 2 then lays out the rank path's scratch and,
// behind it, the per-block bounds and segments (LongScratch); precision 0 only the latter, over blocks of at most
// WR_LONG_BLOCK_ROWS rows.
extern "C" size_t wr_eval_scratch_bytes_topk_long(int64_t R, int64_t n_items, int D, int precision, int k) {
    if (R <= 0 || n_items <= 0 || k < 1 || k > WR_LONG_KMAX) return 0;
    if (precision == 0) {
        if (D != 16 && D != 32 && D != 64 && D != 128 && D != 256) return 0;
        return 1024 + LongScratch::bytes(R < WR_LONG_BLOCK_ROWS ? R : WR_LONG_BLOCK_ROWS);
    }
    if (precision != 2 || (D != 64 && D != 128 && D != 256)) return 0;
    return 1024 + wr_eval_scratch_bytes(R, n_items, D, 2) + LongScratch::bytes(exact_blocking_long(R, n_items));
}

// precision-1 / precision-2 body of wr_eval_rank_topk (eval_kernels.cu dispatches here) and precision 2 of
// wr_eval_rank_topk_long (long_lists: k <= 256, `scratch` past the long call's header)
int wr_eval_rank_tc(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos, int64_t R,
                    int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr, const int32_t *hist_idx,
                    int32_t *rank, float *target, const float *target_in, float *scores_out, int k, int32_t *topk_idx,
                    float *topk_val, void *scratch, WrWorkspace *ws, cudaStream_t st, int precision, bool long_lists) {
    if (D != 64 && D != 128 && D != 256) return WR_E_DIM;
    if (!scratch) return WR_E_NULL;
    if ((reinterpret_cast<uintptr_t>(scratch) & 1023u) != 0) return WR_E_ALIGN;
    const bool exact = precision == 2;
    if (exact && scores_out) return WR_E_TOPK;          // no dense score dump at precision 2
    const int K = exact ? 3 * D : D;
    const int KA = tc_a_cols(D, exact);
    uint8_t *base = static_cast<uint8_t *>(scratch);
    __nv_bfloat16 *A = reinterpret_cast<__nv_bfloat16 *>(base);
    base += align_up((size_t)R * KA * 2, 1024);
    __nv_bfloat16 *Bm = reinterpret_cast<__nv_bfloat16 *>(base);
    base += align_up((size_t)n_items * K * 2, 1024);
    uint8_t *row_ok = base;
    base += align_up((size_t)R, 1024);

    // rows per CTA / items per tile: 128 x 256; 256 x 128 is the measured alternative (WR_TC_VARIANT=12)
    const int mt = (!exact && !topk_idx && tc_variant() == 12) ? 2 : 1;
    const int BMc = TC_BM * mt, BNc = mt == 2 ? 128 : TC_BN;
    CUtensorMap ma, mb;
    int rc = make_map(&mb, Bm, n_items, K, BNc);
    if (rc) return rc;
    TcParams p{};
    p.user = user; p.pos = pos; p.R = R; p.n_users = n_users; p.n_items = n_items;
    p.hist_ptr = hist_ptr; p.hist_idx = hist_idx; p.target = target_in ? target_in : target; p.row_ok = row_ok;
    p.rank = rank; p.scores = scores_out; p.splits = 1; p.k = k; p.top_trigger = k <= 16 ? 4 : 16;    // small k: keep tau fresh
    p.topk_idx = topk_idx; p.topk_val = topk_val;
    if (const char *e = getenv("WR_TC_TOP_TRIGGER")) p.top_trigger = atoi(e);     // tuning knob, <= TC_TOPBUF - 32
    p.n_tiles = (int)((n_items + BNc - 1) / BNc);

    if (!exact) {
        const int64_t n4 = n_items * D / 4;
        pack_items_bf16_kernel<<<(int)min((int64_t)8 * kSMs, (n4 + 255) / 256), 256, 0, st>>>(Iemb, n4, Bm);
        WR_CHECK_LAUNCH();
        if (target_in)
            pack_rows_kernel<<<(int)min((int64_t)8 * kSMs, (R + 7) / 8), 256, 0, st>>>(Uemb, user, R, n_users, D, A, row_ok, ws);
        else
            pack_users_kernel<<<(int)min((int64_t)8 * kSMs, (R + 7) / 8), 256, 0, st>>>(Uemb, Iemb, user, pos, R, n_users,
                                                                                        n_items, D, A, target, row_ok, ws);
        WR_CHECK_LAUNCH();
        rc = make_map(&ma, A, R, K, TC_BM);
        if (rc) return rc;
        const int64_t row_tiles64 = (R + BMc - 1) / BMc;
        if (row_tiles64 > INT32_MAX) return WR_E_SIZE;
        const int row_tiles = (int)row_tiles64;
        int splits = 1;
        // few rows: split the item range over CTAs, one CTA per SM (512 TMEM columns each); rank counts merge with
        // integer atomics.  Top-k lists are per CTA, so that mode keeps a row's items in one CTA.
        if (row_tiles < kSMs && !topk_idx) splits = (kSMs + row_tiles - 1) / row_tiles;
        if (splits > p.n_tiles) splits = p.n_tiles;
        if (splits > 65535) splits = 65535;
        p.tiles_per_split = (p.n_tiles + splits - 1) / splits;
        p.splits = (p.n_tiles + p.tiles_per_split - 1) / p.tiles_per_split;
        if (p.splits > 1) {
            fill_rank_kernel<<<(int)min((int64_t)kSMs * 4, (R + 255) / 256), 256, 0, st>>>(rank, R, 1);
            WR_CHECK_LAUNCH();
        }
        switch (D) {
            case 64: return launch_tc<64>(ma, mb, p, row_tiles, st);
            case 128: return launch_tc<128>(ma, mb, p, row_tiles, st);
            default: return launch_tc<256>(ma, mb, p, row_tiles, st);
        }
    }

    // ---------------- precision 2 ----------------
    float *anorm = reinterpret_cast<float *>(base);
    base += align_up((size_t)R * 4, 1024);
    uint32_t *bmax_bits = reinterpret_cast<uint32_t *>(base);
    unsigned long long *cand_cnt = reinterpret_cast<unsigned long long *>(base + 16);
    base += 1024;
    uint2 *cand = reinterpret_cast<uint2 *>(base);
    int64_t rb;
    unsigned long long cap;
    exact_blocking_topk(R, n_items, topk_idx && !long_lists ? k : 0, &rb, &cap);
    if (long_lists) rb = exact_blocking_long(R, n_items);
    // top-k: per-row candidate counts and segments behind the list (wr_eval_scratch_bytes_topk); long lists: LongScratch
    const size_t seg_at = align_up((size_t)(base - static_cast<uint8_t *>(scratch)) + (size_t)cap * 8, 1024);
    int32_t *seg_cnt = reinterpret_cast<int32_t *>(static_cast<uint8_t *>(scratch) + seg_at);
    int32_t *seg = reinterpret_cast<int32_t *>(static_cast<uint8_t *>(scratch) + seg_at + align_up((size_t)rb * 4, 1024));
    const LongScratch lg(static_cast<uint8_t *>(scratch) + seg_at, rb);
    cudaError_t e = cudaMemsetAsync(bmax_bits, 0, 64, st);
    if (e != cudaSuccess) return (int)e;
    pack_items_split_kernel<<<(int)min((int64_t)16 * kSMs, (n_items + 7) / 8), 256, 0, st>>>(Iemb, n_items, D, Bm, bmax_bits);
    WR_CHECK_LAUNCH();
    pack_users_split_kernel<<<(int)min((int64_t)16 * kSMs, (R + 7) / 8), 256, 0, st>>>(
        Uemb, Iemb, user, pos, R, n_users, n_items, D, target_in ? 1 : 0, exact_a_hilo(D) ? 1 : 0, A, target, anorm, row_ok,
        ws);
    WR_CHECK_LAUNCH();
    p.bmax = reinterpret_cast<const float *>(bmax_bits);
    p.band_c = exact_band_c(D);
    p.cand = cand;
    p.cand_cnt = cand_cnt;
    p.cand_cap = cap;
    p.status = &ws->status;
    for (int64_t r0 = 0; r0 < R; r0 += rb) {
        const int64_t rn = R - r0 < rb ? R - r0 : rb;
        TcParams q = p;
        q.user = user + r0; q.pos = pos + r0; q.R = rn; q.target = p.target + r0; q.row_ok = row_ok + r0; q.rank = rank + r0;
        q.anorm = anorm + r0;
        if (topk_idx) {
            q.topk_idx = topk_idx + r0 * k;
            q.topk_val = topk_val + r0 * k;
            q.seg = seg;
            q.seg_cnt = seg_cnt;
        }
        rc = make_map(&ma, A + r0 * KA, rn, KA, TC_BM);
        if (rc) return rc;
        const int row_tiles = (int)((rn + BMc - 1) / BMc);
        int splits = 1;
        if (row_tiles < kSMs && !topk_idx) splits = (kSMs + row_tiles - 1) / row_tiles;     // lists: one CTA per row
        if (splits > q.n_tiles) splits = q.n_tiles;
        if (splits > 65535) splits = 65535;
        q.tiles_per_split = (q.n_tiles + splits - 1) / splits;
        q.splits = (q.n_tiles + q.tiles_per_split - 1) / q.tiles_per_split;
        if (q.splits > 1) {
            fill_rank_kernel<<<(int)min((int64_t)kSMs * 4, (rn + 255) / 256), 256, 0, st>>>(q.rank, rn, 1);
            WR_CHECK_LAUNCH();
        }
        int ranges = 0, need = 1;
        if (long_lists) {
            // bound pass: the k'-th best t of each item range (its ranks land in the segment counts and are not used)
            int tpr = 0, kp = 0;
            ranges = long_ranges(q.n_tiles, k, &tpr, &kp, &need);
            if (ranges > 0) {
                TcParams b = q;
                b.k = kp;
                b.splits = ranges;
                b.tiles_per_split = tpr;
                b.rank = lg.seg_cnt;
                b.bound = lg.bound;
                e = cudaMemsetAsync(cand_cnt, 0, sizeof(unsigned long long), st);
                if (e != cudaSuccess) return (int)e;
                switch (D) {
                    case 64: rc = launch_tc_v<192, 1, 2, 1, 1, 1>(ma, mb, b, row_tiles, st); break;
                    case 128: rc = launch_tc_v<384, 1, 2, 1, 1, 1>(ma, mb, b, row_tiles, st); break;
                    default: rc = launch_tc_v<768, 1, 2, 1, 1, 1>(ma, mb, b, row_tiles, st); break;
                }
                if (rc) return rc;
            }
        }
        e = cudaMemsetAsync(cand_cnt, 0, sizeof(unsigned long long), st);
        if (e != cudaSuccess) return (int)e;
        if (long_lists) {            // collect pass: the ranks, and every item at or above the row's fixed threshold
            q.k = 1;
            q.seg = lg.seg;
            q.seg_cnt = lg.seg_cnt;
            q.bound = lg.bound;
            q.n_bounds = ranges;
            q.bound_need = need;
            switch (D) {
                case 64: rc = launch_tc_v<192, 1, 2, 1, 1, 2>(ma, mb, q, row_tiles, st); break;
                case 128: rc = launch_tc_v<384, 1, 2, 1, 1, 2>(ma, mb, q, row_tiles, st); break;
                default: rc = launch_tc_v<768, 1, 2, 1, 1, 2>(ma, mb, q, row_tiles, st); break;
            }
        } else if (topk_idx) {       // the ranks as below, plus the drain warps' candidate segments
            switch (D) {
                case 64: rc = launch_tc_v<192, 1, 2, 1, 1>(ma, mb, q, row_tiles, st); break;
                case 128: rc = launch_tc_v<384, 1, 2, 1, 1>(ma, mb, q, row_tiles, st); break;
                default: rc = launch_tc_v<768, 1, 2, 1, 1>(ma, mb, q, row_tiles, st); break;
            }
        } else {
            switch (D) {
                case 64: rc = launch_tc_v<192, 1, 0, 1, 1>(ma, mb, q, row_tiles, st); break;
                case 128: rc = launch_tc_v<384, 1, 0, 1, 1>(ma, mb, q, row_tiles, st); break;
                default: rc = launch_tc_v<768, 1, 0, 1, 1>(ma, mb, q, row_tiles, st); break;       // A_HILO
            }
        }
        if (rc) return rc;
        const float *Ublk = target_in ? Uemb + r0 * D : Uemb;
        eval_recheck_kernel<<<8 * kSMs, 256, 0, st>>>(cand, cand_cnt, cap, Ublk, q.user, target_in ? 1 : 0, Iemb, D,
                                                       q.target, q.rank);
        WR_CHECK_LAUNCH();
        if (long_lists) {
            uint32_t *fallback = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(scratch) - 1024);     // header word 0
            LongSelect sel{lg.seg, lg.seg_cnt, rn, Ublk, q.user, target_in ? 1 : 0, Iemb, D, n_items, hist_ptr, hist_idx, k,
                           topk_idx + r0 * k, topk_val + r0 * k, fallback, &ws->status};
            rc = long_select(sel, st);
            if (rc) return rc;
        } else if (topk_idx) {
            eval_topk_select_kernel<<<(int)min((int64_t)16 * kSMs, (rn + 7) / 8), 256, 0, st>>>(
                seg, seg_cnt, rn, Ublk, q.user, target_in ? 1 : 0, Iemb, D, k, q.topk_idx, q.topk_val, &ws->status);
            WR_CHECK_LAUNCH();
        }
    }
    return WR_OK;
}
