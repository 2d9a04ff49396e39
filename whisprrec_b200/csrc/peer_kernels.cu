// One 8 x B200 box: peer-memory slabs, the cross-GPU barrier (+ small all-reduce), and the row movers that read
// rows from their owning GPU over NVLink.  See the "row-sharded tables" section of include/whisprrec_b200.h.
#include <cmath>
#include <cstring>

#include "common.cuh"

namespace wr {

struct PeerPtrs {
    uint32_t *flags[WR_MAX_WORLD];
    float *slots[WR_MAX_WORLD];
};

__device__ __forceinline__ void st_release_sys_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_f32(float *p, float v) {
    asm volatile("st.relaxed.sys.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ float ld_relaxed_sys_f32(const float *p) {
    float v;
    asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}

// One CTA of 32 threads; thread g talks to rank g.  Deposit the values, publish this rank's arrival in every
// rank's flag array (release at system scope: the stream's earlier kernels have completed, so their peer writes are
// ordered before it), then wait until every rank's arrival for this epoch is visible here.
__global__ void peer_barrier_kernel(PeerPtrs pp, int world, int rank, uint32_t epoch, const float *values_in,
                                    int n_values, float *sums_out, uint32_t *status) {
    const int g = threadIdx.x;
    const int half = (int)(epoch & 1u) * WR_MAX_WORLD * WR_PEER_VALUES;
    if (g < world) {
        for (int v = 0; v < n_values; ++v)
            st_relaxed_sys_f32(pp.slots[g] + half + rank * WR_PEER_VALUES + v, values_in[v]);
        __threadfence_system();
        st_release_sys_u32(pp.flags[g] + rank, epoch);
        // arrivals are monotonic: a rank that is already one epoch ahead has passed this one
        const uint64_t t0 = global_timer_ns();
        while ((int32_t)(ld_acquire_sys_u32(pp.flags[rank] + g) - epoch) < 0) {
            if (global_timer_ns() - t0 > WR_PEER_TIMEOUT_NS) {      // the peer is gone: do not hang the GPU
                if (status) atomicOr(status, WR_STATUS_PEER_TIMEOUT);
                break;
            }
        }
    }
    __syncthreads();
    if (g < n_values) {
        float t = 0.f;
        for (int r = 0; r < world; ++r) t += ld_relaxed_sys_f32(pp.slots[rank] + half + r * WR_PEER_VALUES + g);
        sums_out[g] = t;
    }
}

template <int WHICH>
__global__ void __launch_bounds__(256) gather_rows_sharded_kernel(wr_shards s, const int64_t *idx, int64_t B, int D,
                                                                   float *out, WrWorkspace *ws) {
    const int D4 = D >> 2;
    const int64_t total = B * D4, n_rows = WHICH == 0 ? s.n_users : s.n_items;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = t / D4;
        const int v = (int)(t - b * D4);
        const int64_t r = idx[b];
        float4 x = f4_zero();
        if ((uint64_t)r < (uint64_t)n_rows)
            x = ldg4((WHICH == 0 ? shard_user_row(s, r, D) : shard_item_row(s, r, D)) + 4 * v);
        else if (v == 0)
            atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
        reinterpret_cast<float4 *>(out)[t] = x;
    }
}

// All-gather of a sharded table by PULL: every peer's shard is streamed over NVLink (128-bit loads, 8 in flight per
// thread) into slot g of the local [world, n4] buffer; the own slot is skipped (readers use the shard in place).
__global__ void __launch_bounds__(256) allgather_shards_kernel(wr_shards s, float4 *__restrict__ dst, int64_t n4) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int g0 = 1; g0 < s.world; ++g0) {
        const int g = (s.rank + g0) % s.world;          // every rank starts with a different peer: links evenly loaded
        const float4 *src = reinterpret_cast<const float4 *>(s.base[g]);
        float4 *out = dst + (int64_t)g * n4;
        int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + 7 * stride < n4; i += 8 * stride) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __ldcs(src + i + u * stride);
#pragma unroll
            for (int u = 0; u < 8; ++u) out[i + u * stride] = v[u];
        }
        for (; i < n4; i += stride) out[i] = __ldcs(src + i);
    }
}

__device__ __forceinline__ float bf16_rn(float x) {
    uint32_t u = __float_as_uint(x);
    if ((u & 0x7f800000u) == 0x7f800000u) return x;       // inf / nan unchanged
    u += 0x7fffu + ((u >> 16) & 1u);
    return __uint_as_float(u & 0xffff0000u);
}

// One thread per row, the same d = 0..D-1 fmaf chain as the fp32 scoring kernel's target (eval_kernels.cu).
__global__ void __launch_bounds__(256) rowdot_kernel(const float *__restrict__ A, const float *__restrict__ Bm, int64_t R,
                                                      int D, float *out) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        const float *a = A + r * D, *b = Bm + r * D;
        float s = 0.f;
        for (int v = 0; v < D; v += 4) {
            const float4 x = ldg4(a + v), y = ldg4(b + v);
            s = fmaf(x.x, y.x, s);
            s = fmaf(x.y, y.y, s);
            s = fmaf(x.z, y.z, s);
            s = fmaf(x.w, y.w, s);
        }
        out[r] = s;
    }
}

// bf16 mode: a warp per row in the order pack_users_kernel (eval_tcgen05.cu) uses for its target -- lane-strided
// fmaf chains over the bf16-rounded operands, then the xor-shuffle tree -- so that a sharded evaluation sees the
// very target score the single-GPU tensor-core path does.
__global__ void __launch_bounds__(256) rowdot_bf16_kernel(const float *__restrict__ A, const float *__restrict__ Bm,
                                                           int64_t R, int D, float *out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < R; r += nwarps) {
        float s = 0.f;
        for (int d = lane; d < D; d += 32) s = fmaf(bf16_rn(A[r * D + d]), bf16_rn(Bm[r * D + d]), s);
        s = warp_sum(s);
        if (lane == 0) out[r] = s;
    }
}

// One thread per row: world sorted lists of k (value desc, id asc on ties) -> the k best, by repeated head picks.
__global__ void __launch_bounds__(128) topk_merge_kernel(const float *__restrict__ val, const int32_t *__restrict__ idx,
                                                          int world, int64_t R, int k, float *out_val, int32_t *out_idx) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        int head[WR_MAX_WORLD];
        for (int g = 0; g < world; ++g) head[g] = 0;
        for (int s = 0; s < k; ++s) {
            int best = -1;
            float bv = -INFINITY;
            int32_t bi = -1;
            for (int g = 0; g < world; ++g) {
                if (head[g] >= k) continue;
                const int64_t o = ((int64_t)g * R + r) * k + head[g];
                const int32_t id = idx[o];
                if (id < 0) continue;
                const float v = val[o];
                if (best < 0 || v > bv || (v == bv && id < bi)) {
                    best = g;
                    bv = v;
                    bi = id;
                }
            }
            if (best >= 0) ++head[best];
            out_val[r * k + s] = best >= 0 ? bv : -INFINITY;
            out_idx[r * k + s] = best >= 0 ? bi : -1;
        }
    }
}

}  // namespace wr

using namespace wr;

extern "C" int wr_peer_alloc(size_t bytes, void **out_dev_ptr) {
    if (!out_dev_ptr) return WR_E_NULL;
    if (bytes == 0) return WR_E_SIZE;
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemset(p, 0, bytes);
    if (e != cudaSuccess) {
        cudaFree(p);
        return (int)e;
    }
    *out_dev_ptr = p;
    return WR_OK;
}

extern "C" int wr_peer_free(void *dev_ptr) { return dev_ptr ? (int)cudaFree(dev_ptr) : WR_E_NULL; }

extern "C" int wr_peer_export(void *dev_ptr, unsigned char host_handle[64]) {
    if (!dev_ptr || !host_handle) return WR_E_NULL;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    return (int)cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(host_handle), dev_ptr);
}

extern "C" int wr_peer_open(const unsigned char host_handle[64], void **out_dev_ptr) {
    if (!host_handle || !out_dev_ptr) return WR_E_NULL;
    cudaIpcMemHandle_t h;
    memcpy(&h, host_handle, sizeof(h));
    return (int)cudaIpcOpenMemHandle(out_dev_ptr, h, cudaIpcMemLazyEnablePeerAccess);
}

extern "C" int wr_peer_close(void *dev_ptr) { return dev_ptr ? (int)cudaIpcCloseMemHandle(dev_ptr) : WR_E_NULL; }

extern "C" int wr_peer_barrier(uint32_t *const host_flags[WR_MAX_WORLD], int world, int rank, uint32_t epoch,
                               float *const host_slots[WR_MAX_WORLD], const float *values_in, int n_values,
                               float *sums_out, void *ws, void *stream) {
    if (!host_flags) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || rank < 0 || rank >= world || epoch == 0) return WR_E_SIZE;
    if (n_values < 0 || n_values > WR_PEER_VALUES) return WR_E_SIZE;
    if (n_values > 0 && (!host_slots || !values_in || !sums_out)) return WR_E_NULL;
    PeerPtrs pp{};
    for (int g = 0; g < world; ++g) {
        if (!host_flags[g] || (n_values > 0 && !host_slots[g])) return WR_E_NULL;
        pp.flags[g] = host_flags[g];
        pp.slots[g] = n_values > 0 ? host_slots[g] : nullptr;
    }
    peer_barrier_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(pp, world, rank, epoch, values_in, n_values, sums_out,
                                                            reinterpret_cast<uint32_t *>(ws));
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_gather_rows_sharded(const wr_shards *host_T, int which, const int64_t *idx, int64_t B, int D,
                                      float *out, void *ws, void *stream) {
    if (!host_T || !idx || !out || !ws) return WR_E_NULL;
    const int rc = wr_check_shards(host_T);
    if (rc) return rc;
    if (B < 0 || (which != 0 && which != 1)) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(out)) return WR_E_ALIGN;
    if (B == 0) return WR_OK;
    int64_t g = (B * (D / 4) + 255) / 256;
    if (g > 8 * kSMs) g = 8 * kSMs;
    cudaStream_t st = (cudaStream_t)stream;
    if (which == 0)
        gather_rows_sharded_kernel<0><<<(int)g, 256, 0, st>>>(*host_T, idx, B, D, out, (WrWorkspace *)ws);
    else
        gather_rows_sharded_kernel<1><<<(int)g, 256, 0, st>>>(*host_T, idx, B, D, out, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_allgather_shards(const wr_shards *host_src, float *dst, int D, void *stream) {
    if (!host_src || !dst) return WR_E_NULL;
    const int rc = wr_check_shards(host_src);
    if (rc) return rc;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(dst)) return WR_E_ALIGN;
    if (host_src->world == 1) return WR_OK;
    const int64_t n4 = (host_src->rows_u_local + host_src->rows_i_local) * (D / 4);
    int64_t g = (n4 + 256 * 8 - 1) / (256 * 8);
    if (g > 16 * kSMs) g = 16 * kSMs;
    if (g < 1) g = 1;
    allgather_shards_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(*host_src, reinterpret_cast<float4 *>(dst), n4);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_rowdot(const float *A, const float *B, int64_t R, int D, int round_bf16, float *out, void *stream) {
    if (!A || !B || !out) return WR_E_NULL;
    if (R <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(A) || !wr_aligned16(B)) return WR_E_ALIGN;
    int64_t g = round_bf16 ? (R + 7) / 8 : (R + 255) / 256;
    if (g > 8 * kSMs) g = 8 * kSMs;
    if (round_bf16)
        rowdot_bf16_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(A, B, R, D, out);
    else
        rowdot_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(A, B, R, D, out);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_topk_merge(const float *val, const int32_t *idx, int world, int64_t R, int k, float *out_val,
                             int32_t *out_idx, void *stream) {
    if (!val || !idx || !out_val || !out_idx) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || R <= 0) return WR_E_SIZE;
    if (k < 1 || k > 32) return WR_E_TOPK;
    int64_t g = (R + 127) / 128;
    if (g > 8 * kSMs) g = 8 * kSMs;
    topk_merge_kernel<<<(int)g, 128, 0, (cudaStream_t)stream>>>(val, idx, world, R, k, out_val, out_idx);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

// the same merge for lists of up to WR_LONG_KMAX entries (the kernel is per row and k-agnostic)
extern "C" int wr_topk_merge_long(const float *val, const int32_t *idx, int world, int64_t R, int k, float *out_val,
                                  int32_t *out_idx, void *stream) {
    if (!val || !idx || !out_val || !out_idx) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || R <= 0) return WR_E_SIZE;
    if (k < 1 || k > WR_LONG_KMAX) return WR_E_TOPK;
    int64_t g = (R + 127) / 128;
    if (g > 8 * kSMs) g = 8 * kSMs;
    topk_merge_kernel<<<(int)g, 128, 0, (cudaStream_t)stream>>>(val, idx, world, R, k, out_val, out_idx);
    WR_CHECK_LAUNCH();
    return WR_OK;
}
