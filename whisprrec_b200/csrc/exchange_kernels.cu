// Row exchange for row-sharded tables: the "all-to-all of indices, all-to-all of embedding rows" of the training step
// (SURVEY.md section 8e) built from POSTED NVLink stores only.
//
// Measured on 8 B200s (profiles/r02_prof_sharded_n8_v1.json): random row gathers that LOAD from peer memory reach
// ~30-80 GB/s per GPU (every row is a TLB miss on a multi-GB peer mapping and a 3.5 us round trip), while streaming
// peer stores run at NVLink bandwidth.  So nobody reads remote rows any more:
//   1. wr_xchg_request  every rank buckets the rows its batch slice needs by owner and writes, per owner, the list of
//                       owner-local row indices (+ the role of each: user / positive / negative) into the owner's
//                       request array -- 4 bytes per row;
//      wr_peer_barrier
//   2. wr_xchg_serve    every owner reads the requested rows from its LOCAL shard and stores them, one 128-bit store per
//                       lane, into the requester's receive buffer (dense per owner, in request order);
//      wr_peer_barrier
//   3. the batch kernels run on local memory (wr_bpr_fwd_bwd_exchanged); gradient rows travel the same way in the other
//      direction (the owners' inboxes, wr_inbox_scatter).
// The request lists double as the owner's record of which of its rows the batch touches, once per occurrence -- exactly
// what EmbLoss needs (wr_embloss_owner_*: sums of squares and gradient of the ego rows computed by their owner, no
// traffic at all).
#include "common.cuh"

namespace wr {

struct XchgPtrs {
    int32_t *req[WR_MAX_WORLD];
    uint32_t *req_cnt[WR_MAX_WORLD];
};

// one thread per (batch entry, role)
__global__ void __launch_bounds__(256) xchg_request_kernel(const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B,
                                                            int64_t n_users, int64_t n_items, int world, int rank,
                                                            int64_t rows_u_local, XchgPtrs px, int64_t cap, uint32_t *cnt_local,
                                                            int32_t *where, WrWorkspace *ws) {
    const int64_t total = 3 * B;
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < total; s += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = s / 3;
        const int which = (int)(s - 3 * b);
        const int64_t u = user[b], i = pos[b], j = neg[b];
        const int64_t id = which == 0 ? u : (which == 1 ? i : j);
        // an entry with any id out of range is skipped whole, as the batch kernels skip it: none of its rows is requested
        // (the owners' EmbLoss reads the request lists, so a requested row would count in the norms)
        const bool ok = (uint64_t)u < (uint64_t)n_users && (uint64_t)i < (uint64_t)n_items && (uint64_t)j < (uint64_t)n_items;
        if (!ok) {
            atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
            where[s] = 0;                 // a valid slot (the compute kernel skips the entry by its id check)
            continue;
        }
        const uint32_t q = (uint32_t)id / (uint32_t)world, o = (uint32_t)id - q * (uint32_t)world;
        const int64_t local_row = (which == 0 ? 0 : rows_u_local) + (int64_t)q;
        const uint32_t k = atomicAdd(cnt_local + o, 1u);
        if ((int64_t)k >= cap) {
            atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
            where[s] = 0;
            continue;
        }
        where[s] = (int32_t)((int64_t)o * cap + k);
        px.req[o][(int64_t)rank * cap + k] = (int32_t)((local_row << 2) | which);
    }
}

__global__ void xchg_publish_counts_kernel(XchgPtrs px, int world, int rank, uint32_t *cnt_local) {
    const int o = threadIdx.x;
    if (o < world) {
        px.req_cnt[o][rank] = cnt_local[o];
        cnt_local[o] = 0;                 // ready for the next step
    }
}

struct RecvPtrs {
    float *recv[WR_MAX_WORLD];
};

// a warp per request: one local row -> the requester's receive slot
__global__ void __launch_bounds__(256) xchg_serve_kernel(const float *__restrict__ T, int D, int world, int rank,
                                                          const int32_t *__restrict__ req, const uint32_t *__restrict__ req_cnt,
                                                          int64_t cap, RecvPtrs pr) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int D4 = D >> 2;
    for (int r0 = 0; r0 < world; ++r0) {
        const int r = (rank + r0) % world;                   // requesters visited in a rotated order: links evenly loaded
        const int64_t n = req_cnt[r];
        const int32_t *lst = req + (int64_t)r * cap;
        float *dst = pr.recv[r] + (int64_t)rank * cap * D;
        for (int64_t k = warp; k < n; k += nwarps) {
            const int64_t row = (int64_t)(__ldg(lst + k) >> 2);
            const float *src = T + row * D;
            for (int v = lane; v < D4; v += 32)
                *reinterpret_cast<float4 *>(dst + k * D + 4 * v) = ldg4(src + 4 * v);
        }
    }
}

// EmbLoss on the owner side (utils/loss.py:83-98 as called at LightGCN.py:165-175): the request lists hold every
// occurrence of every ego row of the batch that this rank owns, with its role.
__global__ void __launch_bounds__(256) embloss_owner_sumsq_kernel(const float *__restrict__ T, int D, int world,
                                                                   const int32_t *__restrict__ req,
                                                                   const uint32_t *__restrict__ req_cnt, int64_t cap,
                                                                   float *sumsq_out, WrWorkspace *ws) {
    __shared__ float red[8];
    __shared__ bool flag;
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int D4 = D >> 2;
    float s[3] = {0.f, 0.f, 0.f};
    for (int r = 0; r < world; ++r) {
        const int64_t n = req_cnt[r];
        const int32_t *lst = req + (int64_t)r * cap;
        for (int64_t k = warp; k < n; k += nwarps) {
            const int32_t e = __ldg(lst + k);
            const float *src = T + (int64_t)(e >> 2) * D;
            float a = 0.f;
            for (int v = lane; v < D4; v += 32) {
                const float4 x = ldg4(src + 4 * v);
                a += dot4(x, x);
            }
            const int which = e & 3;
            s[0] += which == 0 ? a : 0.f;
            s[1] += which == 1 ? a : 0.f;
            s[2] += which == 2 ? a : 0.f;
        }
    }
    const float b0 = block_sum(s[0], red), b1 = block_sum(s[1], red), b2 = block_sum(s[2], red);
    if (threadIdx.x == 0) {
        ws->partial[0 * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = b0;
        ws->partial[1 * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = b1;
        ws->partial[2 * WR_MAX_PARTIAL_BLOCKS + blockIdx.x] = b2;
    }
    if (last_block_arrives(&ws->ticket[1], &flag)) {
        if (threadIdx.x < 32) {
            float t[3] = {0.f, 0.f, 0.f};
            for (int i = threadIdx.x; i < (int)gridDim.x; i += 32)
#pragma unroll
                for (int q = 0; q < 3; ++q) t[q] += __ldcg(&ws->partial[q * WR_MAX_PARTIAL_BLOCKS + i]);
#pragma unroll
            for (int q = 0; q < 3; ++q) t[q] = warp_sum(t[q]);
            if (threadIdx.x == 0) {
                sumsq_out[0] = t[0];
                sumsq_out[1] = t[1];
                sumsq_out[2] = t[2];
            }
        }
    }
}

__global__ void __launch_bounds__(256) embloss_owner_scatter_kernel(const float *__restrict__ T, float *G, int D, int world,
                                                                     const int32_t *__restrict__ req,
                                                                     const uint32_t *__restrict__ req_cnt, int64_t cap,
                                                                     float reg_weight, float inv_rows,
                                                                     const float *__restrict__ sumsq_global, float *loss_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int D4 = D >> 2;
    const float k0 = reg_weight * inv_rows;
    const float nu = sqrtf(sumsq_global[0]), np_ = sqrtf(sumsq_global[1]), nn = sqrtf(sumsq_global[2]);
    if (loss_out && blockIdx.x == 0 && threadIdx.x == 0) loss_out[0] += reg_weight * ((nu + np_ + nn) * inv_rows);
    const float kw[3] = {nu > 0.f ? k0 / nu : 0.f, np_ > 0.f ? k0 / np_ : 0.f, nn > 0.f ? k0 / nn : 0.f};
    for (int r = 0; r < world; ++r) {
        const int64_t n = req_cnt[r];
        const int32_t *lst = req + (int64_t)r * cap;
        for (int64_t k = warp; k < n; k += nwarps) {
            const int32_t e = __ldg(lst + k);
            const int64_t row = (int64_t)(e >> 2);
            const int which = e & 3;
            const float c = which == 0 ? kw[0] : (which == 1 ? kw[1] : kw[2]);
            for (int v = lane; v < D4; v += 32) red_add_v4(G + row * D + 4 * v, scale4(ldg4(T + row * D + 4 * v), c));
        }
    }
}

// Sparse all-gather of a row-sharded table that is zero outside the rows of `node_bits` (bitmap over the GLOBAL node
// ids; the pooled gradient of a batch): each owner stores just its marked rows into every peer's copy of its shard.
// A warp looks at 32 local rows at a time; posted NVLink stores only.
__global__ void __launch_bounds__(256) push_marked_rows_kernel(const float *__restrict__ X, wr_shards lay, int D,
                                                                const uint32_t *__restrict__ node_bits, RecvPtrs dst,
                                                                int n_dst) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t n_local = lay.rows_u_local + lay.rows_i_local;
    const int D4 = D >> 2;
    for (int64_t base = warp * 32; base < n_local; base += nwarps * 32) {
        const int64_t lr = base + lane;
        bool set = false;
        if (lr < n_local) {
            int64_t node;
            bool valid;
            if (lr < lay.rows_u_local) {
                node = lr * lay.world + lay.rank;
                valid = node < lay.n_users;
            } else {
                const int64_t it = (lr - lay.rows_u_local) * lay.world + lay.rank;
                node = lay.n_users + it;
                valid = it < lay.n_items;
            }
            set = valid && ((__ldg(node_bits + (node >> 5)) >> (node & 31)) & 1u);
        }
        uint32_t live = __ballot_sync(0xffffffffu, set);
        while (live) {
            const int src = __ffs(live) - 1;
            live &= live - 1;
            const int64_t off = (base + src) * D;
            for (int v = lane; v < D4; v += 32) {
                const float4 x = ldg4(X + off + 4 * v);
                for (int g = 0; g < n_dst; ++g) *reinterpret_cast<float4 *>(dst.recv[g] + off + 4 * v) = x;
            }
        }
    }
}

}  // namespace wr

using namespace wr;

extern "C" int wr_xchg_request(const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B, int64_t n_users,
                               int64_t n_items, int world, int rank, int32_t *const host_req[WR_MAX_WORLD],
                               uint32_t *const host_req_cnt[WR_MAX_WORLD], int64_t cap, uint32_t *cnt_local, int32_t *where,
                               void *ws, void *stream) {
    if (!user || !pos || !neg || !host_req || !host_req_cnt || !cnt_local || !where || !ws) return WR_E_NULL;
    if (B <= 0 || n_users <= 0 || n_items <= 0 || world < 1 || world > WR_MAX_WORLD || rank < 0 || rank >= world ||
        cap < 3 * B || (int64_t)world * cap >= INT32_MAX)
        return WR_E_SIZE;
    const int64_t rows_u_local = (n_users + world - 1) / world, rows_i_local = (n_items + world - 1) / world;
    if (rows_u_local + rows_i_local >= ((int64_t)1 << 29)) return WR_E_SIZE;
    XchgPtrs px;
    for (int g = 0; g < WR_MAX_WORLD; ++g) {
        px.req[g] = g < world ? host_req[g] : nullptr;
        px.req_cnt[g] = g < world ? host_req_cnt[g] : nullptr;
        if (g < world && (!px.req[g] || !px.req_cnt[g])) return WR_E_NULL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int64_t g = (3 * B + 255) / 256;
    if (g > 8 * (int64_t)kSMs) g = 8 * (int64_t)kSMs;
    xchg_request_kernel<<<(int)g, 256, 0, st>>>(user, pos, neg, B, n_users, n_items, world, rank, rows_u_local, px, cap,
                                                 cnt_local, where, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    xchg_publish_counts_kernel<<<1, 32, 0, st>>>(px, world, rank, cnt_local);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_xchg_serve(const float *T_local, int D, int world, int rank, const int32_t *req_local,
                             const uint32_t *req_cnt_local, int64_t cap, float *const host_recv[WR_MAX_WORLD], void *stream) {
    if (!T_local || !req_local || !req_cnt_local || !host_recv) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || rank < 0 || rank >= world || cap <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(T_local)) return WR_E_ALIGN;
    RecvPtrs pr;
    for (int g = 0; g < WR_MAX_WORLD; ++g) {
        pr.recv[g] = g < world ? host_recv[g] : nullptr;
        if (g < world && !pr.recv[g]) return WR_E_NULL;
        if (g < world && !wr_aligned16(pr.recv[g])) return WR_E_ALIGN;
    }
    xchg_serve_kernel<<<16 * kSMs, 256, 0, (cudaStream_t)stream>>>(T_local, D, world, rank, req_local, req_cnt_local, cap, pr);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_embloss_owner_sumsq(const float *T_local, int D, int world, const int32_t *req_local,
                                      const uint32_t *req_cnt_local, int64_t cap, float *sumsq_out, void *ws, void *stream) {
    if (!T_local || !req_local || !req_cnt_local || !sumsq_out || !ws) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || cap <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    embloss_owner_sumsq_kernel<<<4 * kSMs, 256, 0, (cudaStream_t)stream>>>(T_local, D, world, req_local, req_cnt_local, cap,
                                                                          sumsq_out, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_embloss_owner_scatter(const float *T_local, float *G_local, int D, int world, const int32_t *req_local,
                                        const uint32_t *req_cnt_local, int64_t cap, float reg_weight, int64_t B_global,
                                        const float *sumsq_global, float *loss_out, void *stream) {
    if (!T_local || !G_local || !req_local || !req_cnt_local || !sumsq_global) return WR_E_NULL;
    if (world < 1 || world > WR_MAX_WORLD || cap <= 0 || B_global <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(T_local) || !wr_aligned16(G_local)) return WR_E_ALIGN;
    embloss_owner_scatter_kernel<<<8 * kSMs, 256, 0, (cudaStream_t)stream>>>(T_local, G_local, D, world, req_local, req_cnt_local,
                                                                            cap, reg_weight, 1.0f / (float)B_global,
                                                                            sumsq_global, loss_out);
    WR_CHECK_LAUNCH();
    return WR_OK;
}

extern "C" int wr_push_marked_rows(const wr_shards *host_X, int D, const uint32_t *node_bits,
                                   float *const host_push[WR_MAX_WORLD], void *stream) {
    if (!host_X || !node_bits || !host_push) return WR_E_NULL;
    const int rc = wr_check_shards(host_X);
    if (rc) return rc;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    RecvPtrs pr{};
    int n = 0;
    for (int g = 0; g < host_X->world; ++g) {
        if (g == host_X->rank || !host_push[g]) continue;
        if (!wr_aligned16(host_push[g])) return WR_E_ALIGN;
        pr.recv[n++] = host_push[g];
    }
    if (n == 0) return WR_OK;
    const int64_t n_local = host_X->rows_u_local + host_X->rows_i_local;
    int64_t grid = (n_local + 255) / 256;
    if (grid > 16 * kSMs) grid = 16 * kSMs;
    if (grid < 1) grid = 1;
    push_marked_rows_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(host_X->base[host_X->rank], *host_X, D, node_bits, pr, n);
    WR_CHECK_LAUNCH();
    return WR_OK;
}
