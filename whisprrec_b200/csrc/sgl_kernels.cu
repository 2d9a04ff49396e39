// SGL (SURVEY.md section 8 f-3; reference models/general/SGL.py:165-246): the pieces the LightGCN kernels do not cover.
//   * the sum-form BPR term  sum_b -logsigmoid(s+ - s-)  is wr_bpr_logsig_sum_fwd_bwd (train_kernels.cu);
//   * InfoNCE between the two augmented views (SGL.py:196-231), forward and backward, for one block of rows (the users
//     of the batch against all users, or the positive items against all items):
//         a_b = normalize(T1[idx_b]),  t_j = normalize(T2[j]),  e_bj = exp(a_b . t_j / tau),  z_b = sum_j e_bj
//         loss += w * sum_b (log z_b - a_b . t_{idx_b} / tau)
//     The [B, N] contraction runs as fp32 FMA tiles (the parity bar is 1e-5 relative to the reference's fp32 matmul) and
//     is streamed: no buffer grows with B x N, so the table can be any size.
//         pass 1: tiles of s = A T^T / tau in registers, exp, per-(row, table range) partial sums  ->  z, loss
//         pass 2: the same tiles again, W = exp(s) / z  ->  Gt = W^T A (one CTA owns a table tile) and Ga = W T (REDs)
//     8 B N D flop against 6 B N D for a stored W.  Then the chain rule through the two normalisations into the pooled
//     tables' gradients.  exp is taken without a max shift, as the reference does.
#include <algorithm>

#include "common.cuh"

namespace wr {

// ---- out[r] = x / max(||x||, 1e-12) (F.normalize), inv[r] = 1 / max(||x||, 1e-12); x = T[idx ? idx[r] : r] ----
__global__ void __launch_bounds__(256) rows_normalize_kernel(const float *__restrict__ T, const int64_t *idx, int64_t n,
                                                              int64_t n_table, int D, float *out, float *inv, WrWorkspace *ws) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < n; r += nwarps) {
        int64_t src = idx ? idx[r] : r;
        const bool ok = (uint64_t)src < (uint64_t)n_table;
        if (!ok) {
            if (lane == 0) atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
            src = 0;
        }
        const float *x = T + src * D;
        float ss = 0.f;
        for (int d = lane; d < D; d += 32) ss = fmaf(x[d], x[d], ss);
        ss = warp_sum(ss);
        const float k = ok ? 1.0f / fmaxf(sqrtf(ss), 1e-12f) : 0.f;
        for (int d = lane; d < D; d += 32) out[r * D + d] = x[d] * k;
        if (lane == 0) inv[r] = k;
    }
}

// ---- streamed InfoNCE: 64 x 64 tiles of s = A T^T / tau, never stored.  Both operand tiles sit in shared memory as
//      rows [64][DT + 4] (zero past row n and past column D); each thread owns rows ty + 16 i and table rows tx + 16 j
//      and runs the d = 0 .. D-1 fmaf chain of sgemm-style FMA tiles (the padding adds exact zeros). ----
constexpr int IT = 64;                  // rows of a batch tile and of a table tile
constexpr int WR_INFONCE_DMAX = 256;    // both 64-row operand tiles of pass 2 stay in shared memory
constexpr int LDW = IT + 4;             // row stride of the two weight tiles
constexpr int IN_ORDER_BTILES = 8;      // a batch of fewer tiles is neither cut nor rotated in pass 2 (infonce_plan)

__device__ __forceinline__ void cp_async16_zfill(void *smem, const void *gmem, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(valid ? 16 : 0) : "memory");
}

// dst[r][0 .. DT) = src[row0 + r][0 .. D) for r < 64, zero past n rows / D columns (cp.async, caller commits and waits)
template <int DT>
__device__ __forceinline__ void tile_load(float *dst, const float *__restrict__ src, int64_t row0, int64_t n, int D) {
    constexpr int V = DT / 4, LD = DT + 4;
    for (int c = threadIdx.x; c < IT * V; c += blockDim.x) {
        const int r = c / V, v = c - r * V;
        const bool ok = row0 + r < n && 4 * v < D;
        cp_async16_zfill(dst + r * LD + 4 * v, ok ? src + (row0 + r) * D + 4 * v : src, ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int DT>
__device__ __forceinline__ void score_tile(float (&acc)[4][4], const float *sA, const float *sT, int tx, int ty) {
    constexpr int LD = DT + 4;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 4
    for (int v = 0; v < DT / 4; ++v) {
        float4 a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4 *>(sA + (ty + 16 * i) * LD + 4 * v);
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4 *>(sT + (tx + 16 * j) * LD + 4 * v);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
                acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
                acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
                acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
            }
    }
}

template <int CW>
__device__ __forceinline__ void lds_vec(float (&x)[CW], const float *p) {
    if constexpr (CW == 4) {
        const float4 v = *reinterpret_cast<const float4 *>(p);
        x[0] = v.x, x[1] = v.y, x[2] = v.z, x[3] = v.w;
    } else if constexpr (CW == 2) {
        const float2 v = *reinterpret_cast<const float2 *>(p);
        x[0] = v.x, x[1] = v.y;
    } else {
        x[0] = p[0];
    }
}

template <int DT>
constexpr size_t infonce_pass1_smem() { return (size_t)3 * IT * (DT + 4) * 4; }
template <int DT>
constexpr size_t infonce_pass2_smem() { return (size_t)2 * IT * (DT + 4) * 4 + (size_t)2 * IT * LDW * 4; }

// ---- pass 1: part1[r * B + b] = sum over table range r of exp(s_bj) (fixed order); CTA = (batch tile, table range),
//      the table tiles of the range double-buffered ----
template <int DT>
__global__ void __launch_bounds__(256) infonce_pass1_kernel(const float *__restrict__ An, const float *__restrict__ Tn,
                                                             int64_t B, int64_t N, int D, float inv_tau, int tiles_per_range,
                                                             float *part1) {
    constexpr int LD = DT + 4;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sA = reinterpret_cast<float *>(smem_raw), *sT = sA + IT * LD;     // sT: [2][IT][LD]
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t b0 = (int64_t)blockIdx.x * IT;
    const int64_t n_tiles = (N + IT - 1) / IT;
    const int64_t t0 = (int64_t)blockIdx.y * tiles_per_range, t1 = min(n_tiles, t0 + tiles_per_range);
    tile_load<DT>(sA, An, b0, B, D);
    tile_load<DT>(sT, Tn, t0 * IT, N, D);
    float rs[4] = {0.f, 0.f, 0.f, 0.f};
    for (int64_t t = t0; t < t1; ++t) {
        const int buf = (int)((t - t0) & 1);
        if (t + 1 < t1) {
            tile_load<DT>(sT + (buf ^ 1) * IT * LD, Tn, (t + 1) * IT, N, D);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        float acc[4][4];
        score_tile<DT>(acc, sA, sT + buf * IT * LD, tx, ty);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool live = t * IT + tx + 16 * j < N;
#pragma unroll
            for (int i = 0; i < 4; ++i) rs[i] += live ? expf(inv_tau * acc[i][j]) : 0.f;
        }
        __syncthreads();                                         // buffer buf is refilled next iteration
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float v = rs[i];
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);    // the 16 lanes of one ty
        const int64_t b = b0 + ty + 16 * i;
        if (tx == 0 && b < B) part1[blockIdx.y * B + b] = v;
    }
}

// ---- z_b = sum_r part1[r][b] (fixed order), iz_b = 1 / z_b, part[b] = log z_b - a_b . t_{idx_b} / tau; one warp a row ----
__global__ void __launch_bounds__(256) infonce_rows_kernel(const float *__restrict__ part1, int n_ranges, int64_t Bn, int64_t N,
                                                            const float *__restrict__ An, const float *__restrict__ Tn,
                                                            const int64_t *idx, int D, float inv_tau, float *iz, float *part) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t b = warp; b < Bn; b += nwarps) {
        float z = 0.f;
        for (int r = lane; r < n_ranges; r += 32) z += part1[r * Bn + b];
        z = warp_sum(z);
        int64_t t = idx[b];
        if ((uint64_t)t >= (uint64_t)N) t = 0;                   // flagged by rows_normalize_kernel
        float p = 0.f;
        for (int d = lane; d < D; d += 32) p = fmaf(An[b * D + d], Tn[t * D + d], p);
        p = warp_sum(p);
        if (lane == 0) {
            iz[b] = 1.0f / z;
            part[b] = logf(z) - p * inv_tau;
        }
    }
}

// ---- pass 2: W_bj = exp(s_bj) / z_b recomputed per tile; CTA = (table tile, range of batch tiles):
//        Gt_j = sum_b W_bj a_b in registers over the range, stored once into Gtp[q] (q = 0 is Gt itself);
//        Ga_b += sum_j W_bj t_j as one RED per element and tile pair.
//      Thread (tx, ty) owns rows ty + 16 i of each output and columns (tx + 16 k) CW + v. ----
template <int DT>
__global__ void __launch_bounds__(256) infonce_pass2_kernel(const float *__restrict__ An, const float *__restrict__ Tn,
                                                             const float *__restrict__ iz, int64_t B, int64_t N, int D,
                                                             float inv_tau, int tiles_per_range, float *Ga, float *Gt,
                                                             float *Gtp) {
    constexpr int LD = DT + 4;
    constexpr int CW = DT >= 64 ? 4 : DT / 16, NK = DT / (16 * CW);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sT = reinterpret_cast<float *>(smem_raw), *sA = sT + IT * LD;
    float *sWt = sA + IT * LD;      // [b][4 y + i] = W[b][y + 16 i]   (Gt reads 4 table rows of one batch row)
    float *sWg = sWt + IT * LDW;    // [j][4 y + i] = W[y + 16 i][j]   (Ga reads 4 batch rows of one table row)
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t j0 = (int64_t)blockIdx.x * IT;
    const int64_t n_btiles = (B + IT - 1) / IT;
    const int64_t q0 = (int64_t)blockIdx.y * tiles_per_range, q1 = min(n_btiles, q0 + tiles_per_range);
    const int64_t nq = q1 - q0;
    float gt[4][NK][CW];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < NK; ++k)
#pragma unroll
            for (int v = 0; v < CW; ++v) gt[i][k][v] = 0.f;
    // on a batch of IN_ORDER_BTILES tiles or more, table tiles start at different batch tiles so that their REDs into Ga
    // do not meet on the same rows; a smaller batch is walked from its first tile
    const int64_t first = (nq > 0 && n_btiles >= IN_ORDER_BTILES) ? (int64_t)blockIdx.x % nq : 0;
    tile_load<DT>(sT, Tn, j0, N, D);
    if (nq > 0) tile_load<DT>(sA, An, (q0 + first) * IT, B, D);
    for (int64_t s = 0; s < nq; ++s) {
        const int64_t b0 = (q0 + (first + s) % nq) * IT;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        float acc[4][4];
        score_tile<DT>(acc, sA, sT, tx, ty);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t b = b0 + ty + 16 * i;
            const float izb = b < B ? iz[b] : 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                acc[i][j] = (b < B && j0 + tx + 16 * j < N) ? expf(inv_tau * acc[i][j]) * izb : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
            *reinterpret_cast<float4 *>(sWt + (ty + 16 * i) * LDW + 4 * tx) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4 *>(sWg + (tx + 16 * j) * LDW + 4 * ty) = make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]);
        __syncthreads();
        // Gt[j0 + ty + 16 i][c] += sum_b W[b][j] A[b][c]
#pragma unroll 4
        for (int b = 0; b < IT; ++b) {
            const float4 w = *reinterpret_cast<const float4 *>(sWt + b * LDW + 4 * ty);
            const float wi[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < NK; ++k) {
                float a[CW];
                lds_vec<CW>(a, sA + b * LD + (tx + 16 * k) * CW);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int v = 0; v < CW; ++v) gt[i][k][v] = fmaf(wi[i], a[v], gt[i][k][v]);
            }
        }
        __syncthreads();                                         // sA is free: fetch the next batch tile under the Ga work
        if (s + 1 < nq) tile_load<DT>(sA, An, (q0 + (first + s + 1) % nq) * IT, B, D);
        // Ga[b0 + ty + 16 i][c] += sum_j W[b][j] T[j][c]
        float ga[4][NK][CW];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < NK; ++k)
#pragma unroll
                for (int v = 0; v < CW; ++v) ga[i][k][v] = 0.f;
#pragma unroll 4
        for (int j = 0; j < IT; ++j) {
            const float4 w = *reinterpret_cast<const float4 *>(sWg + j * LDW + 4 * ty);
            const float wi[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < NK; ++k) {
                float t[CW];
                lds_vec<CW>(t, sT + j * LD + (tx + 16 * k) * CW);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int v = 0; v < CW; ++v) ga[i][k][v] = fmaf(wi[i], t[v], ga[i][k][v]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t b = b0 + ty + 16 * i;
            if (b >= B) continue;
#pragma unroll
            for (int k = 0; k < NK; ++k) {
                const int c = (tx + 16 * k) * CW;
                if (c >= D) continue;
                float *dst = Ga + b * D + c;
                if constexpr (CW == 4) atomicAdd(reinterpret_cast<float4 *>(dst), make_float4(ga[i][k][0], ga[i][k][1], ga[i][k][2], ga[i][k][3]));
                else if constexpr (CW == 2) atomicAdd(reinterpret_cast<float2 *>(dst), make_float2(ga[i][k][0], ga[i][k][1]));
                else atomicAdd(dst, ga[i][k][0]);
            }
        }
    }
    float *out = blockIdx.y == 0 ? Gt : Gtp + (int64_t)(blockIdx.y - 1) * N * D;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t j = j0 + ty + 16 * i;
        if (j >= N) continue;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
            const int c = (tx + 16 * k) * CW;
            if (c >= D) continue;
#pragma unroll
            for (int v = 0; v < CW; ++v) out[j * D + c + v] = gt[i][k][v];
        }
    }
}

// Gt[e] += Gtp[0][e] + ... + Gtp[n - 1][e], in that order
__global__ void __launch_bounds__(256) infonce_gt_reduce_kernel(float *Gt, const float *__restrict__ Gtp, int n, int64_t len) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < len; e += (int64_t)gridDim.x * blockDim.x) {
        float s = Gt[e];
        for (int q = 0; q < n; ++q) s += Gtp[q * len + e];
        Gt[e] = s;
    }
}

// deterministic sum of part[0 .. n) -> loss_out[0] += w * sum   (one CTA)
__global__ void __launch_bounds__(256) scaled_sum_kernel(const float *__restrict__ part, int64_t n, float w, float *loss_out) {
    __shared__ float red[8];
    float s = 0.f;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += part[i];
    const float t = block_sum(s, red);
    if (threadIdx.x == 0) loss_out[0] += w * t;
}

// ---- batch side: g = c (Ga_b - t_{idx_b}) w.r.t. the normalised a_b, through the normalisation into dT1[idx_b] (RED);
//      the positive pair's pull on t_{idx_b}: Gt[idx_b] -= a_b (RED, before infonce_table_kernel runs) ----
__global__ void __launch_bounds__(256) infonce_batch_kernel(const float *__restrict__ Ga, const float *__restrict__ An,
                                                             const float *__restrict__ inv1, const float *__restrict__ Tn,
                                                             const int64_t *idx, int64_t Bn, int64_t N, int D, float c,
                                                             float *dT1, float *Gt) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t b = warp; b < Bn; b += nwarps) {
        const int64_t t = idx[b];
        if ((uint64_t)t >= (uint64_t)N) continue;               // flagged by rows_normalize_kernel
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) {
            const float g = Ga[b * D + d] - Tn[t * D + d];
            dot = fmaf(g, An[b * D + d], dot);
        }
        dot = warp_sum(dot);
        const float k = c * inv1[b];
        for (int d = lane; d < D; d += 32) {
            const float a = An[b * D + d];
            const float g = Ga[b * D + d] - Tn[t * D + d];
            atomicAdd(dT1 + t * D + d, k * (g - dot * a));
            atomicAdd(Gt + t * D + d, -a);
        }
    }
}

// ---- table side: g = c Gt_j w.r.t. the normalised t_j, through the normalisation, added to dT2[j] ----
__global__ void __launch_bounds__(256) infonce_table_kernel(const float *__restrict__ Gt, const float *__restrict__ Tn,
                                                             const float *__restrict__ inv2, int64_t N, int D, float c, float *dT2) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t j = warp; j < N; j += nwarps) {
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) dot = fmaf(Gt[j * D + d], Tn[j * D + d], dot);
        dot = warp_sum(dot);
        const float k = c * inv2[j];
        for (int d = lane; d < D; d += 32) dT2[j * D + d] += k * (Gt[j * D + d] - dot * Tn[j * D + d]);
    }
}

static inline size_t sgl_align(size_t x) { return (x + 255) & ~(size_t)255; }

// Grid of the two passes.  Pass 1: the table is cut into n_ranges ranges so that batch tiles x ranges fill about four
// waves of CTAs.  Pass 2: one CTA per table tile; only a table of fewer than two tiles per SM also cuts the batch, into at
// most 8 ranges of at least 4 batch tiles, whose Gt partials are summed afterwards (that buffer is at most 7 N D floats
// with N < 128 SMs).  A batch of fewer than IN_ORDER_BTILES tiles is neither cut nor rotated: Gt is then one fmaf chain
// over b = 0 .. B-1 in order, the order of the materialised W^T A product this replaced, which matters where duplicate
// ids make Gt[idx_b] - a_b cancel.
struct InfoncePlan {
    int DT;
    int64_t n_btiles, n_ttiles;
    int64_t tiles_per_range1, n_ranges1, tiles_per_range2, n_ranges2;
};

static InfoncePlan infonce_plan(int64_t B, int64_t N, int D) {
    InfoncePlan p;
    p.DT = D <= 16 ? 16 : D <= 32 ? 32 : D <= 64 ? 64 : D <= 128 ? 128 : 256;
    p.n_btiles = (B + IT - 1) / IT;
    p.n_ttiles = (N + IT - 1) / IT;
    const int64_t sms = kSMs;
    int64_t r = std::min(p.n_ttiles, std::max<int64_t>(1, (4 * sms + p.n_btiles - 1) / p.n_btiles));
    p.tiles_per_range1 = (p.n_ttiles + r - 1) / r;
    p.n_ranges1 = (p.n_ttiles + p.tiles_per_range1 - 1) / p.tiles_per_range1;
    int64_t q = std::min(std::max<int64_t>(1, std::min(p.n_btiles / (IN_ORDER_BTILES / 2), (int64_t)8)),
                         std::max<int64_t>(1, (2 * sms + p.n_ttiles - 1) / p.n_ttiles));
    p.tiles_per_range2 = (p.n_btiles + q - 1) / q;
    p.n_ranges2 = (p.n_btiles + p.tiles_per_range2 - 1) / p.tiles_per_range2;
    return p;
}

template <int DT>
static int infonce_pass1_launch(const InfoncePlan &pl, const float *An, const float *Tn, int64_t B, int64_t N, int D,
                                float inv_tau, float *part1, cudaStream_t st) {
    const size_t s1 = infonce_pass1_smem<DT>();
    cudaError_t e = cudaFuncSetAttribute(infonce_pass1_kernel<DT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1);
    if (e != cudaSuccess) return (int)e;
    infonce_pass1_kernel<DT><<<dim3((unsigned)pl.n_btiles, (unsigned)pl.n_ranges1), 256, s1, st>>>(
        An, Tn, B, N, D, inv_tau, (int)pl.tiles_per_range1, part1);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

template <int DT>
static int infonce_pass2_launch(const InfoncePlan &pl, const float *An, const float *Tn, const float *iz, int64_t B,
                                int64_t N, int D, float inv_tau, float *Ga, float *Gt, float *Gtp, cudaStream_t st) {
    const size_t s2 = infonce_pass2_smem<DT>();
    cudaError_t e = cudaFuncSetAttribute(infonce_pass2_kernel<DT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2);
    if (e != cudaSuccess) return (int)e;
    infonce_pass2_kernel<DT><<<dim3((unsigned)pl.n_ttiles, (unsigned)pl.n_ranges2), 256, s2, st>>>(
        An, Tn, iz, B, N, D, inv_tau, (int)pl.tiles_per_range2, Ga, Gt, Gtp);
    WR_CHECK_LAUNCH();
    if (pl.n_ranges2 > 1) {
        const int64_t len = N * D;
        infonce_gt_reduce_kernel<<<(int)std::min((int64_t)8 * kSMs, (len + 255) / 256), 256, 0, st>>>(Gt, Gtp, (int)pl.n_ranges2 - 1, len);
        WR_CHECK_LAUNCH();
    }
    return WR_OK;
}

static int infonce_pass1(const InfoncePlan &pl, const float *An, const float *Tn, int64_t B, int64_t N, int D,
                         float inv_tau, float *part1, cudaStream_t st) {
    switch (pl.DT) {
        case 16: return infonce_pass1_launch<16>(pl, An, Tn, B, N, D, inv_tau, part1, st);
        case 32: return infonce_pass1_launch<32>(pl, An, Tn, B, N, D, inv_tau, part1, st);
        case 64: return infonce_pass1_launch<64>(pl, An, Tn, B, N, D, inv_tau, part1, st);
        case 128: return infonce_pass1_launch<128>(pl, An, Tn, B, N, D, inv_tau, part1, st);
        default: return infonce_pass1_launch<256>(pl, An, Tn, B, N, D, inv_tau, part1, st);
    }
}

static int infonce_pass2(const InfoncePlan &pl, const float *An, const float *Tn, const float *iz, int64_t B, int64_t N,
                         int D, float inv_tau, float *Ga, float *Gt, float *Gtp, cudaStream_t st) {
    switch (pl.DT) {
        case 16: return infonce_pass2_launch<16>(pl, An, Tn, iz, B, N, D, inv_tau, Ga, Gt, Gtp, st);
        case 32: return infonce_pass2_launch<32>(pl, An, Tn, iz, B, N, D, inv_tau, Ga, Gt, Gtp, st);
        case 64: return infonce_pass2_launch<64>(pl, An, Tn, iz, B, N, D, inv_tau, Ga, Gt, Gtp, st);
        case 128: return infonce_pass2_launch<128>(pl, An, Tn, iz, B, N, D, inv_tau, Ga, Gt, Gtp, st);
        default: return infonce_pass2_launch<256>(pl, An, Tn, iz, B, N, D, inv_tau, Ga, Gt, Gtp, st);
    }
}

// ---- InfoNCE split by table shard (wr_infonce_sharded_*): every rank runs the global batch against its own rows ----
struct PeerSlots {
    float *p[WR_MAX_WORLD];    // p[g]: rank g's slot array as mapped here
    int world;
};

// z_b of this rank's rows = sum_r part1[r][b] (r ascending), posted into slot [rank][b] of every rank's [world][B] array
// (plain stores: the wr_peer_barrier that follows orders them before any reader)
__global__ void __launch_bounds__(256) infonce_post_partials_kernel(const float *__restrict__ part1, int n_ranges, int64_t B,
                                                                     PeerSlots z, int world, int rank) {
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int r = 0; r < n_ranges; ++r) s += part1[r * B + b];
        for (int g = 0; g < world; ++g) z.p[g][rank * B + b] = s;
    }
}

// the positive pair's pull, applied by the owner of idx_b only: Gt[local(idx_b)] -= a_b (RED: duplicate ids)
__global__ void __launch_bounds__(256) infonce_owner_pull_kernel(const float *__restrict__ An, const int64_t *idx, int64_t Bn,
                                                                  int64_t n_rows, int D, int world, int rank, float *Gt) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t b = warp; b < Bn; b += nwarps) {
        const int64_t t = idx[b];
        if ((uint64_t)t >= (uint64_t)n_rows || t % world != rank) continue;
        const int64_t l = t / world;
        for (int d = lane; d < D; d += 32) atomicAdd(Gt + l * D + d, -An[b * D + d]);
    }
}

// this rank's partial Ga_b, stored into slot [rank][b] of the owner of idx_b ([world][B][D] per rank)
__global__ void __launch_bounds__(256) infonce_post_ga_kernel(const float *__restrict__ Ga, const int64_t *idx, int64_t Bn,
                                                               int64_t n_rows, int D, PeerSlots ga, int rank) {
    const int D4 = D >> 2;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < Bn * D4; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / D4;
        const int v = (int)(e - b * D4);
        const int64_t t = idx[b];
        if ((uint64_t)t >= (uint64_t)n_rows) continue;
        float *dst = ga.p[t % ga.world] + ((int64_t)rank * Bn + b) * D + 4 * v;
        *reinterpret_cast<float4 *>(dst) = reinterpret_cast<const float4 *>(Ga + b * D)[v];
    }
}

// owner side of the batch: Ga_b = sum over ranks r (ascending) of slot [r][b]; then infonce_batch_kernel's chain rule
// through the normalisation of a_b into the local row of dT1 (RED: duplicate ids)
__global__ void __launch_bounds__(256) infonce_owner_batch_kernel(const float *__restrict__ ga_local, int world, int rank,
                                                                   const float *__restrict__ An, const float *__restrict__ inv1,
                                                                   const float *__restrict__ Pn, const int64_t *idx,
                                                                   int64_t Bn, int64_t n_rows, int D, float c, float *dT1) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t b = warp; b < Bn; b += nwarps) {
        const int64_t t = idx[b];
        if ((uint64_t)t >= (uint64_t)n_rows || t % world != rank) continue;
        const int64_t l = t / world;
        auto g_at = [&](int d) {
            float s = 0.f;
            for (int r = 0; r < world; ++r) s += ga_local[((int64_t)r * Bn + b) * D + d];
            return s - Pn[b * D + d];
        };
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) dot = fmaf(g_at(d), An[b * D + d], dot);
        dot = warp_sum(dot);
        const float k = c * inv1[b];
        for (int d = lane; d < D; d += 32) atomicAdd(dT1 + l * D + d, k * (g_at(d) - dot * An[b * D + d]));
    }
}

__global__ void iota_kernel(int64_t *out, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = i;
}

// Scratch of one rank, carried from phase to phase: its table rows (Tn, Gt, inv2, Gtp) and the whole batch's rows.
struct InfonceShardScratch {
    InfoncePlan pl;
    float *Tn, *Gt, *inv2, *An, *Pn, *Ga, *inv1, *iz, *part, *part1, *Gtp;
    int64_t *iota;
};

static size_t infonce_shard_layout(int64_t B, int64_t N_local, int D, void *scratch, InfonceShardScratch *s) {
    // an empty shard plans as one row (never launched), so the layout is defined for every rank
    const int64_t N = std::max<int64_t>(N_local, 1);
    InfonceShardScratch t;
    t.pl = infonce_plan(B, N, D);
    char *p = (char *)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    char *const p0 = p;
    auto take = [&](size_t bytes) { char *q = p; p += sgl_align(bytes); return q; };
    t.Tn = (float *)take((size_t)N * D * 4), t.Gt = (float *)take((size_t)N * D * 4), t.inv2 = (float *)take((size_t)N * 4);
    t.An = (float *)take((size_t)B * D * 4), t.Pn = (float *)take((size_t)B * D * 4), t.Ga = (float *)take((size_t)B * D * 4);
    t.inv1 = (float *)take((size_t)B * 4), t.iz = (float *)take((size_t)B * 4), t.part = (float *)take((size_t)B * 4);
    t.iota = (int64_t *)take((size_t)B * 8);
    t.part1 = (float *)take((size_t)t.pl.n_ranges1 * B * 4);
    t.Gtp = (float *)take((size_t)(t.pl.n_ranges2 - 1) * N * D * 4);
    if (s) *s = t;
    return (size_t)(p - p0) + 256;
}

}  // namespace wr

using namespace wr;

extern "C" size_t wr_infonce_scratch_bytes(int64_t B, int64_t N, int D) {
    if (B <= 0 || N <= 0 || D <= 0 || D > WR_INFONCE_DMAX) return 0;
    const InfoncePlan pl = infonce_plan(B, N, D);
    return sgl_align((size_t)N * D * 4) * 2 /* Tn, Gt */ + sgl_align((size_t)N * 4) /* inv2 */ +
           sgl_align((size_t)B * D * 4) * 2 /* An, Ga */ + sgl_align((size_t)B * 4) * 3 /* inv1, iz, part */ +
           sgl_align((size_t)pl.n_ranges1 * B * 4) /* part1 */ + sgl_align((size_t)(pl.n_ranges2 - 1) * N * D * 4) /* Gtp */ +
           256;
}

extern "C" int wr_infonce_fwd_bwd(const float *T1, const float *T2, const int64_t *idx, int64_t B, int64_t N, int D,
                                  float tau, float weight, float grad_scale, float *dT1, float *dT2, float *loss_out,
                                  void *scratch, size_t scratch_bytes, void *ws, void *stream) {
    if (!T1 || !T2 || !idx || !dT1 || !dT2 || !loss_out || !scratch || !ws) return WR_E_NULL;
    if (B <= 0 || N <= 0 || tau <= 0.f) return WR_E_SIZE;
    if (D <= 0 || (D & 3) || D > WR_INFONCE_DMAX) return WR_E_DIM;
    if (scratch_bytes < wr_infonce_scratch_bytes(B, N, D)) return WR_E_SIZE;
    cudaStream_t st = (cudaStream_t)stream;
    const InfoncePlan pl = infonce_plan(B, N, D);
    char *p = (char *)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    auto take = [&](size_t bytes) { char *q = p; p += sgl_align(bytes); return q; };
    float *Tn = (float *)take((size_t)N * D * 4), *Gt = (float *)take((size_t)N * D * 4), *inv2 = (float *)take((size_t)N * 4);
    float *An = (float *)take((size_t)B * D * 4), *Ga = (float *)take((size_t)B * D * 4);
    float *inv1 = (float *)take((size_t)B * 4), *iz = (float *)take((size_t)B * 4), *part = (float *)take((size_t)B * 4);
    float *part1 = (float *)take((size_t)pl.n_ranges1 * B * 4);
    float *Gtp = (float *)take((size_t)(pl.n_ranges2 - 1) * N * D * 4);
    const float inv_tau = 1.0f / tau;
    const int gw = 8 * kSMs;
    rows_normalize_kernel<<<(int)min((int64_t)gw, (N + 7) / 8), 256, 0, st>>>(T2, nullptr, N, N, D, Tn, inv2, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    rows_normalize_kernel<<<(int)min((int64_t)gw, (B + 7) / 8), 256, 0, st>>>(T1, idx, B, N, D, An, inv1, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    cudaError_t e = cudaMemsetAsync(Ga, 0, (size_t)B * D * 4, st);
    if (e != cudaSuccess) return (int)e;
    int rc = infonce_pass1(pl, An, Tn, B, N, D, inv_tau, part1, st);
    if (rc != WR_OK) return rc;
    infonce_rows_kernel<<<(int)std::min((int64_t)8 * kSMs, (B + 7) / 8), 256, 0, st>>>(part1, (int)pl.n_ranges1, B, N, An, Tn,
                                                                                     idx, D, inv_tau, iz, part);
    WR_CHECK_LAUNCH();
    rc = infonce_pass2(pl, An, Tn, iz, B, N, D, inv_tau, Ga, Gt, Gtp, st);
    if (rc != WR_OK) return rc;
    scaled_sum_kernel<<<1, 256, 0, st>>>(part, B, weight, loss_out);
    WR_CHECK_LAUNCH();
    const float c = weight * inv_tau * grad_scale;
    infonce_batch_kernel<<<(int)min((int64_t)gw, (B + 7) / 8), 256, 0, st>>>(Ga, An, inv1, Tn, idx, B, N, D, c, dT1, Gt);
    WR_CHECK_LAUNCH();
    infonce_table_kernel<<<(int)min((int64_t)gw, (N + 7) / 8), 256, 0, st>>>(Gt, Tn, inv2, N, D, c, dT2);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

// ---- InfoNCE split by table shard -------------------------------------------------------------------------------------
// Block `which` (0: users, 1: items) of the pooled view tables; this rank's block rows are local rows off .. off + N_local
// of its shard (global id = l * world + rank), the rest of the block's rows (padding) never enter z.
struct InfonceShardArgs {
    int64_t n_rows, N_local, off;
};

static int infonce_shard_args(const wr_shards *s, int which, int64_t B, int D, float tau, float *const host_slots[WR_MAX_WORLD],
                              bool need16, InfonceShardArgs *a) {
    const int rc = wr_check_shards(s);
    if (rc) return rc;
    if (which != 0 && which != 1) return WR_E_SIZE;
    if (B <= 0 || !(tau > 0.f)) return WR_E_SIZE;
    if (D <= 0 || (D & 3) || D > WR_INFONCE_DMAX) return WR_E_DIM;
    for (int g = 0; g < s->world; ++g) {
        if (!host_slots[g]) return WR_E_NULL;
        if (need16 && !wr_aligned16(host_slots[g])) return WR_E_ALIGN;
    }
    a->n_rows = which == 0 ? s->n_users : s->n_items;
    a->N_local = s->rank < a->n_rows ? (a->n_rows - s->rank + s->world - 1) / s->world : 0;
    a->off = which == 0 ? 0 : s->rows_u_local;
    return WR_OK;
}

static PeerSlots peer_slots(float *const host_slots[WR_MAX_WORLD], int world) {
    PeerSlots p{};
    for (int g = 0; g < world; ++g) p.p[g] = host_slots[g];
    p.world = world;
    return p;
}

extern "C" size_t wr_infonce_sharded_scratch_bytes(int64_t B, int64_t N_local, int D) {
    if (B <= 0 || N_local < 0 || D <= 0 || (D & 3) || D > WR_INFONCE_DMAX) return 0;
    return infonce_shard_layout(B, N_local, D, nullptr, nullptr);
}

extern "C" int wr_infonce_sharded_partials(const wr_shards *host_T1, const wr_shards *host_T2, int which, const int64_t *idx,
                                           int64_t B, int D, float tau, float *const host_z[WR_MAX_WORLD], void *scratch,
                                           size_t scratch_bytes, void *ws, void *stream) {
    if (!host_T1 || !host_T2 || !idx || !host_z || !scratch || !ws) return WR_E_NULL;
    InfonceShardArgs a;
    int rc = wr_check_shards(host_T1);
    if (rc) return rc;
    rc = infonce_shard_args(host_T2, which, B, D, tau, host_z, false, &a);
    if (rc) return rc;
    if (host_T1->world != host_T2->world || host_T1->rank != host_T2->rank) return WR_E_SIZE;
    if (scratch_bytes < wr_infonce_sharded_scratch_bytes(B, a.N_local, D)) return WR_E_SIZE;
    InfonceShardScratch s;
    infonce_shard_layout(B, a.N_local, D, scratch, &s);
    cudaStream_t st = (cudaStream_t)stream;
    const int gw = 8 * kSMs;
    const float inv_tau = 1.0f / tau;
    iota_kernel<<<(int)min((int64_t)gw, (B + 255) / 256), 256, 0, st>>>(s.iota, B);
    WR_CHECK_LAUNCH();
    // the batch's rows of both views from their owners (Ga holds the raw rows until phase 2 clears it)
    rc = wr_gather_rows_sharded(host_T1, which, idx, B, D, s.Ga, ws, stream);
    if (rc) return rc;
    rows_normalize_kernel<<<(int)min((int64_t)gw, (B + 7) / 8), 256, 0, st>>>(s.Ga, nullptr, B, B, D, s.An, s.inv1, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    rc = wr_gather_rows_sharded(host_T2, which, idx, B, D, s.Ga, ws, stream);
    if (rc) return rc;
    rows_normalize_kernel<<<(int)min((int64_t)gw, (B + 7) / 8), 256, 0, st>>>(s.Ga, nullptr, B, B, D, s.Pn, s.iz, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    if (a.N_local > 0) {
        const float *T2l = host_T2->base[host_T2->rank] + a.off * D;
        rows_normalize_kernel<<<(int)min((int64_t)gw, (a.N_local + 7) / 8), 256, 0, st>>>(T2l, nullptr, a.N_local, a.N_local, D,
                                                                                         s.Tn, s.inv2, (WrWorkspace *)ws);
        WR_CHECK_LAUNCH();
        rc = infonce_pass1(s.pl, s.An, s.Tn, B, a.N_local, D, inv_tau, s.part1, st);
        if (rc) return rc;
    }
    infonce_post_partials_kernel<<<(int)min((int64_t)gw, (B + 255) / 256), 256, 0, st>>>(
        s.part1, a.N_local > 0 ? (int)s.pl.n_ranges1 : 0, B, peer_slots(host_z, host_T2->world), host_T2->world, host_T2->rank);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_infonce_sharded_weights(const wr_shards *host_dT2, int which, const int64_t *idx, int64_t B, int D,
                                          float tau, float weight, float grad_scale, float *const host_z[WR_MAX_WORLD],
                                          float *const host_ga[WR_MAX_WORLD], float *loss_out, void *scratch,
                                          size_t scratch_bytes, void *stream) {
    if (!host_dT2 || !idx || !host_z || !host_ga || !loss_out || !scratch) return WR_E_NULL;
    InfonceShardArgs a;
    int rc = infonce_shard_args(host_dT2, which, B, D, tau, host_z, false, &a);
    if (rc) return rc;
    rc = infonce_shard_args(host_dT2, which, B, D, tau, host_ga, true, &a);
    if (rc) return rc;
    if (scratch_bytes < wr_infonce_sharded_scratch_bytes(B, a.N_local, D)) return WR_E_SIZE;
    InfonceShardScratch s;
    infonce_shard_layout(B, a.N_local, D, scratch, &s);
    cudaStream_t st = (cudaStream_t)stream;
    const int gw = 8 * kSMs, world = host_dT2->world, rank = host_dT2->rank;
    const float inv_tau = 1.0f / tau;
    // z_b from the world partials (the same bits on every rank), the loss rows against the gathered positives
    infonce_rows_kernel<<<(int)std::min((int64_t)gw, (B + 7) / 8), 256, 0, st>>>(host_z[rank], world, B, B, s.An, s.Pn, s.iota,
                                                                                D, inv_tau, s.iz, s.part);
    WR_CHECK_LAUNCH();
    scaled_sum_kernel<<<1, 256, 0, st>>>(s.part, B, weight, loss_out);
    WR_CHECK_LAUNCH();
    cudaError_t e = cudaMemsetAsync(s.Ga, 0, (size_t)B * D * 4, st);
    if (e != cudaSuccess) return (int)e;
    if (a.N_local > 0) {
        rc = infonce_pass2(s.pl, s.An, s.Tn, s.iz, B, a.N_local, D, inv_tau, s.Ga, s.Gt, s.Gtp, st);
        if (rc) return rc;
        infonce_owner_pull_kernel<<<(int)min((int64_t)gw, (B + 7) / 8), 256, 0, st>>>(s.An, idx, B, a.n_rows, D, world, rank, s.Gt);
        WR_CHECK_LAUNCH();
        const float c = weight * inv_tau * grad_scale;
        infonce_table_kernel<<<(int)min((int64_t)gw, (a.N_local + 7) / 8), 256, 0, st>>>(
            s.Gt, s.Tn, s.inv2, a.N_local, D, c, host_dT2->base[rank] + a.off * D);
        WR_CHECK_LAUNCH();
    }
    infonce_post_ga_kernel<<<(int)min((int64_t)gw, (B * (D / 4) + 255) / 256), 256, 0, st>>>(s.Ga, idx, B, a.n_rows, D,
                                                                                           peer_slots(host_ga, world), rank);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_infonce_sharded_batch(const wr_shards *host_dT1, int which, const int64_t *idx, int64_t B, int D,
                                        float tau, float weight, float grad_scale, float *const host_ga[WR_MAX_WORLD],
                                        void *scratch, size_t scratch_bytes, void *stream) {
    if (!host_dT1 || !idx || !host_ga || !scratch) return WR_E_NULL;
    InfonceShardArgs a;
    int rc = infonce_shard_args(host_dT1, which, B, D, tau, host_ga, true, &a);
    if (rc) return rc;
    if (scratch_bytes < wr_infonce_sharded_scratch_bytes(B, a.N_local, D)) return WR_E_SIZE;
    InfonceShardScratch s;
    infonce_shard_layout(B, a.N_local, D, scratch, &s);
    const int world = host_dT1->world, rank = host_dT1->rank;
    const float c = weight * (1.0f / tau) * grad_scale;
    infonce_owner_batch_kernel<<<(int)min((int64_t)8 * kSMs, (B + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        host_ga[rank], world, rank, s.An, s.inv1, s.Pn, idx, B, a.n_rows, D, c, host_dT1->base[rank] + a.off * D);
    WR_CHECK_LAUNCH();
    return WR_OK;
}
