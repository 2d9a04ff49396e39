// Full-ranking evaluation, fp32-exact variant: a register-tiled score kernel whose epilogue applies the
// per-user history mask (bitmask built from the sorted history CSR), counts items that beat the target and
// maintains a per-row top-k -- the [rows, n_items] score matrix of BaseRunner.interface is never written.
#include "common.cuh"

namespace wr {

constexpr int EV_TR = 64;   // eval rows per CTA
constexpr int EV_TI = 64;   // items per tile
constexpr int EV_KMAX = 32;

struct EvalParams {
    const float *Uemb, *Iemb;
    const int64_t *user, *pos;
    int64_t R, n_users, n_items;
    const int64_t *hist_ptr;
    const int32_t *hist_idx;
    int k;
    int32_t *topk_idx;
    float *topk_val;
    int32_t *rank;
    float *target;
    float *scores;  // optional dense [R, n_items] output (unmasked), the reference's full_predict
    int splits, tiles_per_split, n_tiles;
    WrWorkspace *ws;
    // item-shard mode (wr_eval_rank_topk_shard): Uemb holds the R gathered user rows, the target scores are an
    // input (the target item may live on another shard: pos = -1) and `target` is not written
    const float *target_in;
    // long lists (TOPK 2 / 3 below): the k'-th best of each item range per row, and the collected candidates
    float *bound;
    int n_bounds, bound_need;
    int32_t *seg, *seg_cnt;
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Thread (ty, tx) of the 16x16 grid owns rows ty+16i and columns tx+16j (i, j < 4): with a row pitch of D+4
// floats the 128-bit shared loads of a quarter warp then fall into 8 distinct 4-bank groups (no conflicts).
// TOPK: 0 ranks only; 1 the k-best lists (k <= 32); 3 the same lists over item ranges (blockIdx.y), of which only the
// k-th best value is written (p.bound: the bound pass of a long call); 2 every unmasked item scoring at least the row's
// bound is appended to its candidate segment (the collect pass).
// Top-k at D = 256 would need 233,984 B of shared memory with a separate staging buffer S, over the 232,448 B a CTA
// may have: there S takes the B buffer the FMA loop has just consumed (one more barrier per tile).
template <int D, int TOPK>
struct EvalSmem {
    static constexpr int LD = D + 4;
    static constexpr bool S_IN_B = TOPK && D >= 256;
    static constexpr size_t S_BYTES = TOPK && !S_IN_B ? (size_t)EV_TR * (EV_TI + 1) * 4 : 0;
    static constexpr size_t BYTES = (size_t)(EV_TR * LD + 2 * EV_TI * LD) * 4 + 2 * EV_TR * 2 * 4 + EV_TR * 4 + S_BYTES +
                                    (TOPK ? (size_t)EV_TR * EV_KMAX * 8 : 0);
    static_assert(!S_IN_B || EV_TR * (EV_TI + 1) <= EV_TI * LD, "S fits in one B buffer");
    static_assert(BYTES <= 227 * 1024, "shared memory budget");
};

template <int D, int TOPK>
__global__ void __launch_bounds__(256) eval_rank_kernel(EvalParams p) {
    using SM = EvalSmem<D, TOPK>;
    constexpr int LD = SM::LD;
    constexpr int D4 = D / 4;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *As = reinterpret_cast<float *>(smem_raw);            // [EV_TR][LD]
    float *Bs = As + EV_TR * LD;                                 // [2][EV_TI][LD]
    uint32_t *mask = reinterpret_cast<uint32_t *>(Bs + 2 * EV_TI * LD);  // [2][EV_TR][2]
    float *st_s = reinterpret_cast<float *>(mask + 2 * EV_TR * 2);       // [EV_TR]
    float *S = st_s + EV_TR;                                     // [EV_TR][EV_TI+1]     (TOPK only; S_IN_B: per tile)
    float *tkv = S + SM::S_BYTES / 4;                            // [EV_TR][EV_KMAX]     (TOPK only)
    int32_t *tki = reinterpret_cast<int32_t *>(tkv + EV_TR * EV_KMAX);

    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * EV_TR;
    const int t0 = blockIdx.y * p.tiles_per_split;
    const int t1 = min(p.n_tiles, t0 + p.tiles_per_split);

    // ---- user rows of this CTA -> shared (zero rows for r >= R or an out-of-range id) ----
    for (int c = tid; c < EV_TR * D4; c += 256) {
        const int i = c / D4, v = c - i * D4;
        const int64_t r = row0 + i;
        float4 x = f4_zero();
        if (r < p.R) {
            const int64_t u = p.user[r];
            if ((uint64_t)u < (uint64_t)p.n_users) x = ldg4(p.Uemb + (p.target_in ? r : u) * D + 4 * v);
        }
        *reinterpret_cast<float4 *>(As + i * LD + 4 * v) = x;
    }
    auto load_tile = [&](int t, int buf) {
        const int64_t j0 = (int64_t)t * EV_TI;
        float *dst = Bs + buf * EV_TI * LD;
        for (int c = tid; c < EV_TI * D4; c += 256) {
            const int i = c / D4, v = c - i * D4;
            if (j0 + i < p.n_items) cp_async16(dst + i * LD + 4 * v, p.Iemb + (j0 + i) * D + 4 * v);
        }
        cp_async_commit();
    };
    if (t0 < t1) load_tile(t0, 0);
    if (TOPK == 1 || TOPK == 3) {
        for (int c = tid; c < EV_TR * EV_KMAX; c += 256) {
            tkv[c] = -INFINITY;
            tki[c] = -1;
        }
    }
    if (TOPK == 2 && tid < EV_TR) {       // collect: slot 0 holds the row's bound and its candidate count
        const int64_t r = row0 + tid;
        tkv[tid * EV_KMAX] = r < p.R ? long_bound(p.bound + r * WR_LONG_RANGES, p.n_bounds, p.bound_need) : -INFINITY;
        tki[tid * EV_KMAX] = 0;
    }
    __syncthreads();

    // ---- per-row state held by threads 0..63: target score, history cursor ----
    int64_t cur = 0, hend = 0;
    bool row_live = false;
    if (tid < EV_TR) {
        const int64_t r = row0 + tid;
        float st = 0.f;
        if (r < p.R) {
            const int64_t u = p.user[r], it = p.pos[r];
            if ((uint64_t)u < (uint64_t)p.n_users && (p.target_in || (uint64_t)it < (uint64_t)p.n_items)) {
                row_live = true;
                if (p.target_in) {
                    st = p.target_in[r];
                } else {
                    const float *a = As + tid * LD;
                    const float *b = p.Iemb + it * D;
#pragma unroll 4
                    for (int v = 0; v < D4; ++v) {
                        const float4 x = *reinterpret_cast<const float4 *>(a + 4 * v), y = ldg4(b + 4 * v);
                        st = fmaf(x.x, y.x, st);
                        st = fmaf(x.y, y.y, st);
                        st = fmaf(x.z, y.z, st);
                        st = fmaf(x.w, y.w, st);
                    }
                }
                cur = p.hist_ptr[u];
                hend = p.hist_ptr[u + 1];
                // first history entry at or after this CTA's first item
                const int32_t first = (int32_t)min((int64_t)t0 * EV_TI, (int64_t)INT32_MAX);
                int64_t lo = cur, hi = hend;
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (p.hist_idx[mid] < first) lo = mid + 1; else hi = mid;
                }
                cur = lo;
                if (TOPK != 3 && blockIdx.y == 0 && !p.target_in) p.target[r] = st;
            } else {
                atomicOr(&p.ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
            }
        }
        st_s[tid] = st;
    }

    int cnt[4] = {0, 0, 0, 0};
    for (int t = t0; t < t1; ++t) {
        const int buf = (t - t0) & 1;
        const int64_t j0 = (int64_t)t * EV_TI;
        if (t + 1 < t1) load_tile(t + 1, buf ^ 1);
        if (tid < EV_TR) {
            uint32_t m0 = 0, m1 = 0;
            if (!row_live) {
                m0 = m1 = 0xffffffffu;
            } else {
                while (cur < hend) {
                    const int64_t h = (int64_t)p.hist_idx[cur] - j0;
                    if (h >= EV_TI) break;
                    if (h >= 32) m1 |= 1u << (h - 32); else if (h >= 0) m0 |= 1u << h;
                    ++cur;
                }
                const int64_t live = p.n_items - j0;  // columns past the table are masked
                if (live < 32) { m0 |= ~0u << (live < 0 ? 0 : live); m1 = ~0u; }
                else if (live < 64) m1 |= ~0u << (live - 32);
            }
            mask[(buf * EV_TR + tid) * 2 + 0] = m0;
            mask[(buf * EV_TR + tid) * 2 + 1] = m1;
        }
        if (t + 1 < t1) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncthreads();

        const float *Bt = Bs + buf * EV_TI * LD;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 2
        for (int v = 0; v < D4; ++v) {
            float4 a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4 *>(As + (ty + 16 * i) * LD + 4 * v);
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4 *>(Bt + (tx + 16 * j) * LD + 4 * v);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    // the same d = 0..D-1 FMA chain as the target score above: comparisons are consistent
                    acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
                    acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
                    acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
                    acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
                }
        }
        if (SM::S_IN_B) {
            __syncthreads();                                     // every thread is done reading Bt
            S = Bs + buf * EV_TI * LD;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = ty + 16 * i;
            const float st = st_s[rl];
            const uint32_t m0 = mask[(buf * EV_TR + rl) * 2 + 0], m1 = mask[(buf * EV_TR + rl) * 2 + 1];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t word = j < 2 ? m0 : m1;
                const bool masked = (word >> (tx + 16 * (j & 1))) & 1u;
                cnt[i] += (!masked && acc[i][j] > st) ? 1 : 0;
                if (TOPK) S[rl * (EV_TI + 1) + tx + 16 * j] = masked ? -INFINITY : acc[i][j];
                if (p.scores) {
                    const int64_t r = row0 + rl, c = j0 + tx + 16 * j;
                    if (r < p.R && c < p.n_items) p.scores[r * p.n_items + c] = acc[i][j];
                }
            }
        }
        if (TOPK == 2) {
            __syncthreads();
            // warp w appends the tile's items of rows 8w..8w+7 that reach the row's bound, in item order
            for (int q = 0; q < 8; ++q) {
                const int rl = warp * 8 + q;
                const float L = tkv[rl * EV_KMAX];
                int n = tki[rl * EV_KMAX];
                int32_t *segr = p.seg + (row0 + rl) * WR_LONG_SEG_CAP;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float s = S[rl * (EV_TI + 1) + h * 32 + lane];
                    const uint32_t take = __ballot_sync(0xffffffffu, s >= L && s > -INFINITY);
                    const int at = n + __popc(take & ((1u << lane) - 1u));
                    if (((take >> lane) & 1u) && at < WR_LONG_SEG_CAP) segr[at] = (int32_t)(j0 + h * 32 + lane);
                    n += __popc(take);
                }
                __syncwarp();
                if (lane == 0) tki[rl * EV_KMAX] = n;
            }
        }
        if (TOPK == 1 || TOPK == 3) {
            __syncthreads();
            // warp w merges the tile's scores of rows 8w..8w+7 into their sorted lists (lane = list slot)
            const uint32_t kmask = p.k >= 32 ? 0xffffffffu : ((1u << p.k) - 1u);
            for (int q = 0; q < 8; ++q) {
                const int rl = warp * 8 + q;
                float tv = tkv[rl * EV_KMAX + lane];
                int32_t ti = tki[rl * EV_KMAX + lane];
                float tau = __shfl_sync(0xffffffffu, tv, p.k - 1);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float s = S[rl * (EV_TI + 1) + h * 32 + lane];
                    const int32_t id = (int32_t)(j0 + h * 32 + lane);
                    // items arrive in ascending id, so a tie with the k-th best never displaces it
                    uint32_t pend = __ballot_sync(0xffffffffu, s > tau);
                    while (pend) {
                        const int src = __ffs(pend) - 1;
                        pend &= pend - 1;
                        const float v = __shfl_sync(0xffffffffu, s, src);
                        const int32_t vid = __shfl_sync(0xffffffffu, id, src);
                        if (!(v > tau)) continue;
                        const int ins = __popc(__ballot_sync(0xffffffffu, tv >= v) & kmask);
                        const float up_v = __shfl_up_sync(0xffffffffu, tv, 1);
                        const int32_t up_i = __shfl_up_sync(0xffffffffu, ti, 1);
                        if (lane == ins) { tv = v; ti = vid; }
                        else if (lane > ins) { tv = up_v; ti = up_i; }
                        tau = __shfl_sync(0xffffffffu, tv, p.k - 1);
                    }
                }
                tkv[rl * EV_KMAX + lane] = tv;
                tki[rl * EV_KMAX + lane] = ti;
            }
        }
        __syncthreads();
    }

    // ---- ranks: fold the 16 column-threads of each row ----
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int c = cnt[i];
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        const int64_t r = row0 + ty + 16 * i;
        if (TOPK != 3 && tx == 0 && r < p.R) {
            if (p.splits == 1) p.rank[r] = 1 + c;
            else atomicAdd(&p.rank[r], c);
        }
    }
    if (TOPK == 2 && tid < EV_TR && row0 + tid < p.R) p.seg_cnt[row0 + tid] = tki[tid * EV_KMAX];
    if (TOPK == 3 && tid < EV_TR && row0 + tid < p.R)
        p.bound[(row0 + tid) * WR_LONG_RANGES + blockIdx.y] = tkv[tid * EV_KMAX + p.k - 1];
    if (TOPK == 1) {
        for (int c = tid; c < EV_TR * p.k; c += 256) {
            const int i = c / p.k, s = c - i * p.k;
            const int64_t r = row0 + i;
            if (r < p.R) {
                p.topk_idx[r * p.k + s] = tki[i * EV_KMAX + s];
                p.topk_val[r * p.k + s] = tkv[i * EV_KMAX + s];
            }
        }
    }
}

__global__ void fill_i32_kernel(int32_t *x, int64_t n, int32_t v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] = v;
}

// HR@k / NDCG@k sums in float64; per-block partials are added in block order by the last block.
__global__ void __launch_bounds__(256) metrics_kernel(const int32_t *__restrict__ rank, int64_t R, int nk, int k0,
                                                       int k1, int k2, int k3, int k4, int k5, int k6, int k7,
                                                       double *out, WrWorkspace *ws) {
    const int ks[8] = {k0, k1, k2, k3, k4, k5, k6, k7};
    __shared__ double red[8][16];
    __shared__ bool flag;
    double hr[8], nd[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) hr[q] = nd[q] = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < R; i += (int64_t)gridDim.x * blockDim.x) {
        const int rk = rank[i];
        const double gain = 1.0 / log2((double)rk + 1.0);
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (q < nk && rk <= ks[q]) { hr[q] += 1.0; nd[q] += gain; }
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            hr[q] += __shfl_xor_sync(0xffffffffu, hr[q], o);
            nd[q] += __shfl_xor_sync(0xffffffffu, nd[q], o);
        }
        if (lane == 0) { red[w][q] = hr[q]; red[w][8 + q] = nd[q]; }
    }
    __syncthreads();
    if (threadIdx.x < 16) {
        double t = 0.0;
        for (int ww = 0; ww < 8; ++ww) t += red[ww][threadIdx.x];
        ws->dpartial[blockIdx.x * 16 + threadIdx.x] = t;
    }
    if (last_block_arrives(&ws->ticket[2], &flag)) {
        if (threadIdx.x < 16) {
            double t = 0.0;
            for (int b = 0; b < (int)gridDim.x; ++b) t += __ldcg(&ws->dpartial[b * 16 + threadIdx.x]);
            const int q = threadIdx.x & 7;
            if (q < nk) out[(threadIdx.x >> 3) * nk + q] = t / (double)R;
        }
    }
}

template <int D, int TOPK>
static int launch_eval(EvalParams &p, cudaStream_t st, int row_tiles) {
    const size_t smem = EvalSmem<D, TOPK>::BYTES;
    cudaError_t e = cudaFuncSetAttribute(eval_rank_kernel<D, TOPK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid(row_tiles, p.splits);
    eval_rank_kernel<D, TOPK><<<grid, 256, smem, st>>>(p);
    e = cudaGetLastError();
    return (int)e;
}

// precision 0's score: s = fmaf(a_d, b_d, s), d = 0 .. D-1
__device__ __forceinline__ float fma_chain(const float *a, const float *b, int D) {
    float s = 0.f;
    for (int d = 0; d < D; d += 4) {
        const float4 x = ldg4(a + d), y = ldg4(b + d);
        s = fmaf(x.x, y.x, s);
        s = fmaf(x.y, y.y, s);
        s = fmaf(x.z, y.z, s);
        s = fmaf(x.w, y.w, s);
    }
    return s;
}

// One 64-bit key per candidate whose ascending order is (value desc, id asc), the order of top_worse; -inf (masked) and
// NaN scores get the padding key ~0 and never enter a list.  -0 and +0 are one value, so they tie by id.
__device__ __forceinline__ unsigned long long long_key(float s, int32_t id) {
    if (!(s > -INFINITY)) return ~0ull;
    uint32_t u = __float_as_uint(s == 0.f ? 0.f : s);
    u ^= (u >> 31) ? 0xffffffffu : 0x80000000u;              // ascending in the value
    return ((unsigned long long)~u << 32) | (uint32_t)id;
}

// ascending bitonic sort of n (a power of two) keys in shared memory by the whole CTA
__device__ void bitonic_sort(unsigned long long *key, int n) {
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < n / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const unsigned long long a = key[lo], b = key[hi];
                if ((a > b) == ((lo & size) == 0)) {
                    key[lo] = b;
                    key[hi] = a;
                }
            }
            __syncthreads();
        }
}

// Long lists, last pass: one CTA per row.  The row's candidates (every unmasked item at or above its bound, a superset of
// precision 0's top k) are re-scored and sorted; the first k are the list, padded with (-1, -inf).  A row with more than
// WR_LONG_SEG_CAP candidates is finished here too: the CTA scans every item in chunks of WR_LONG_SEG_CAP - k, each
// sorted together with the k best so far, so the sweep cannot overflow.
constexpr int LS_THREADS = 256;
__global__ void __launch_bounds__(LS_THREADS) eval_topk_long_select_kernel(LongSelect q) {
    __shared__ unsigned long long key[WR_LONG_SEG_CAP];
    const int tid = threadIdx.x;
    for (int64_t r = blockIdx.x; r < q.R; r += gridDim.x) {
        const int n = q.seg_cnt[r];
        // rows with candidates had an in-range user (the passes mask every item of the others)
        const float *a = n > 0 ? q.U + (q.rows_gathered ? r : q.user[r]) * q.D : nullptr;
        if (n <= WR_LONG_SEG_CAP) {
            int P = 1;
            while (P < n || P < q.k) P <<= 1;
            for (int i = tid; i < P; i += LS_THREADS) {
                unsigned long long kk = ~0ull;
                if (i < n) {
                    const int32_t id = q.seg[r * WR_LONG_SEG_CAP + i];
                    kk = long_key(fma_chain(a, q.I + (int64_t)id * q.D, q.D), id);
                }
                key[i] = kk;
            }
            __syncthreads();
            bitonic_sort(key, P);
        } else {
            if (tid == 0) {
                atomicAdd(q.fallback, 1u);
                atomicOr(q.status, WR_STATUS_TOPK_OVERFLOW);
            }
            const int64_t u = q.user[r], h0 = q.hist_ptr[u], h1 = q.hist_ptr[u + 1];
            for (int i = tid; i < q.k; i += LS_THREADS) key[i] = ~0ull;
            const int chunk = WR_LONG_SEG_CAP - q.k;
            for (int64_t j0 = 0; j0 < q.n_items; j0 += chunk) {
                for (int i = tid; i < chunk; i += LS_THREADS) {
                    const int64_t j = j0 + i;
                    unsigned long long kk = ~0ull;
                    if (j < q.n_items) {
                        int64_t lo = h0, hi = h1;            // the history is sorted
                        while (lo < hi) {
                            const int64_t mid = (lo + hi) >> 1;
                            if (q.hist_idx[mid] < j) lo = mid + 1; else hi = mid;
                        }
                        if (lo == h1 || q.hist_idx[lo] != j)
                            kk = long_key(fma_chain(a, q.I + j * q.D, q.D), (int32_t)j);
                    }
                    key[q.k + i] = kk;
                }
                __syncthreads();
                bitonic_sort(key, WR_LONG_SEG_CAP);
            }
        }
        for (int s = tid; s < q.k; s += LS_THREADS) {
            const unsigned long long kk = key[s];
            const int32_t id = (int32_t)(uint32_t)kk;
            q.topk_idx[r * q.k + s] = kk == ~0ull ? -1 : id;
            q.topk_val[r * q.k + s] = kk == ~0ull ? -INFINITY : fma_chain(a, q.I + (int64_t)id * q.D, q.D);
        }
        __syncthreads();
    }
}

int long_select(const LongSelect &q, cudaStream_t st) {
    eval_topk_long_select_kernel<<<(int)min((int64_t)16 * kSMs, q.R), LS_THREADS, 0, st>>>(q);
    return (int)cudaGetLastError();
}

}  // namespace wr

using namespace wr;

// eval_tcgen05.cu
int wr_eval_rank_tc(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos, int64_t R,
                    int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr, const int32_t *hist_idx,
                    int32_t *rank, float *target, const float *target_in, float *scores_out, int k, int32_t *topk_idx,
                    float *topk_val, void *scratch, WrWorkspace *ws, cudaStream_t st, int precision, bool long_lists);

static int eval_rank_topk_impl(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos,
                               int64_t R, int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr,
                               const int32_t *hist_idx, int k, int precision, int32_t *topk_idx, float *topk_val,
                               int32_t *rank, float *target, const float *target_in, float *scores_out,
                               void *scratch, void *ws, void *stream) {
    if (!Uemb || !Iemb || !user || !pos || !hist_ptr || !hist_idx || !rank || !ws) return WR_E_NULL;
    if (!target && !target_in) return WR_E_NULL;
    if ((topk_idx == nullptr) != (topk_val == nullptr)) return WR_E_NULL;
    if (R <= 0 || n_users <= 0 || n_items <= 0 || n_items > INT32_MAX - 1024) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (topk_idx && (k < 1 || k > EV_KMAX)) return WR_E_TOPK;
    if (!wr_aligned16(Uemb) || !wr_aligned16(Iemb)) return WR_E_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const bool topk = topk_idx != nullptr;
    if (precision == 1 || precision == 2) {
        return wr_eval_rank_tc(Uemb, Iemb, user, pos, R, n_users, n_items, D, hist_ptr, hist_idx, rank, target,
                               target_in, scores_out, topk ? k : 0, topk_idx, topk_val, scratch, (WrWorkspace *)ws, st,
                               precision, false);
    }
    if (precision != 0) return WR_E_PRECISION;
    EvalParams p{Uemb, Iemb, user, pos, R, n_users, n_items, hist_ptr, hist_idx, topk ? k : 1,
                 topk_idx, topk_val, rank, target, scores_out, 1, 0, 0, (WrWorkspace *)ws, target_in};
    p.n_tiles = (int)((n_items + EV_TI - 1) / EV_TI);
    const int64_t row_tiles64 = (R + EV_TR - 1) / EV_TR;
    if (row_tiles64 > INT32_MAX) return WR_E_SIZE;
    const int row_tiles = (int)row_tiles64;
    // few eval rows: split the item range over CTAs (rank counts merge with integer atomics -> still exact)
    int splits = 1;
    if (!topk && row_tiles < 2 * kSMs) splits = (2 * kSMs + row_tiles - 1) / row_tiles;
    if (splits > p.n_tiles) splits = p.n_tiles;
    if (splits > 65535) splits = 65535;
    p.tiles_per_split = (p.n_tiles + splits - 1) / splits;
    p.splits = (p.n_tiles + p.tiles_per_split - 1) / p.tiles_per_split;
    if (p.splits > 1) {
        fill_i32_kernel<<<(int)min((int64_t)kSMs * 4, (R + 255) / 256), 256, 0, st>>>(rank, R, 1);
        WR_CHECK_LAUNCH();
    }
    int rc;
#define WR_EVAL_CALL(DD) rc = topk ? launch_eval<DD, 1>(p, st, row_tiles) : launch_eval<DD, 0>(p, st, row_tiles)
    switch (D) {
        case 16: WR_EVAL_CALL(16); break;
        case 32: WR_EVAL_CALL(32); break;
        case 64: WR_EVAL_CALL(64); break;
        case 128: WR_EVAL_CALL(128); break;
        case 256: WR_EVAL_CALL(256); break;
        default: return WR_E_DIM;
    }
#undef WR_EVAL_CALL
    return rc;
}

extern "C" int wr_eval_rank_topk(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos,
                                 int64_t R, int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr,
                                 const int32_t *hist_idx, int k, int precision, int32_t *topk_idx, float *topk_val,
                                 int32_t *rank, float *target, float *scores_out, void *scratch, void *ws,
                                 void *stream) {
    if (!target) return WR_E_NULL;
    return eval_rank_topk_impl(Uemb, Iemb, user, pos, R, n_users, n_items, D, hist_ptr, hist_idx, k, precision,
                               topk_idx, topk_val, rank, target, nullptr, scores_out, scratch, ws, stream);
}

extern "C" int wr_eval_rank_topk_shard(const float *Urows, const float *Iemb, const int64_t *user,
                                       const int64_t *pos_local, int64_t R, int64_t n_users, int64_t n_items_local,
                                       int D, const int64_t *hist_ptr, const int32_t *hist_idx, int k, int precision,
                                       const float *target, int32_t *topk_idx, float *topk_val, int32_t *rank,
                                       void *scratch, void *ws, void *stream) {
    if (!target) return WR_E_NULL;
    return eval_rank_topk_impl(Urows, Iemb, user, pos_local, R, n_users, n_items_local, D, hist_ptr, hist_idx, k,
                               precision, topk_idx, topk_val, rank, nullptr, target, nullptr, scratch, ws, stream);
}

// Long lists (k up to 256): precision 2 runs in wr_eval_rank_tc; precision 0 here, per block of rows, in three passes.
//   bound:   eval_rank_kernel<D, 3> over `ranges` item ranges (blockIdx.y) writes the k'-th best score of each range
//   collect: eval_rank_kernel<D, 2> computes the ranks and appends every unmasked item with s >= the row's bound L
//   select:  eval_topk_long_select_kernel sorts the candidates (and sweeps the rows whose segment overflowed)
// The need-th largest bound L is a lower bound on the row's k-th best score (long_bound), so the candidates hold
// precision 0's top k (DESIGN.md section 4.3).
static int eval_rank_topk_long_impl(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos,
                                    int64_t R, int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr,
                                    const int32_t *hist_idx, int k, int precision, int32_t *topk_idx, float *topk_val,
                                    int32_t *rank, float *target, const float *target_in, void *scratch, void *ws,
                                    void *stream) {
    if (!Uemb || !Iemb || !user || !pos || !hist_ptr || !hist_idx || !rank || !ws || !topk_idx || !topk_val)
        return WR_E_NULL;
    if (!target && !target_in) return WR_E_NULL;
    if (!scratch) return WR_E_NULL;
    if (k < 1 || k > WR_LONG_KMAX || (precision != 0 && precision != 2)) return WR_E_TOPK;
    if (R <= 0 || n_users <= 0 || n_items <= 0 || n_items > INT32_MAX - 1024) return WR_E_SIZE;
    if (precision == 0 ? (D != 16 && D != 32 && D != 64 && D != 128 && D != 256) : (D != 64 && D != 128 && D != 256))
        return WR_E_DIM;
    if (!wr_aligned16(Uemb) || !wr_aligned16(Iemb) || (reinterpret_cast<uintptr_t>(scratch) & 1023u) != 0)
        return WR_E_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t *fallback = static_cast<uint32_t *>(scratch);
    cudaError_t e = cudaMemsetAsync(fallback, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess) return (int)e;
    void *body = static_cast<uint8_t *>(scratch) + 1024;
    if (precision == 2)
        return wr_eval_rank_tc(Uemb, Iemb, user, pos, R, n_users, n_items, D, hist_ptr, hist_idx, rank, target, target_in,
                               nullptr, k, topk_idx, topk_val, body, (WrWorkspace *)ws, st, 2, true);

    const int64_t rb = R < WR_LONG_BLOCK_ROWS ? R : WR_LONG_BLOCK_ROWS;
    LongScratch lg(body, rb);
    const int n_tiles = (int)((n_items + EV_TI - 1) / EV_TI);
    int tpr = n_tiles, kp = k, need = 1;
    const int ranges = long_ranges(n_tiles, k, &tpr, &kp, &need);
    for (int64_t r0 = 0; r0 < R; r0 += rb) {
        const int64_t rn = R - r0 < rb ? R - r0 : rb;
        EvalParams p{target_in ? Uemb + r0 * D : Uemb, Iemb, user + r0, pos + r0, rn, n_users, n_items, hist_ptr, hist_idx,
                     1, nullptr, nullptr, rank + r0, target ? target + r0 : nullptr, nullptr, 1, n_tiles, n_tiles,
                     (WrWorkspace *)ws, target_in ? target_in + r0 : nullptr};
        p.bound = lg.bound;
        p.n_bounds = ranges;
        p.bound_need = need;
        p.seg = lg.seg;
        p.seg_cnt = lg.seg_cnt;
        const int row_tiles = (int)((rn + EV_TR - 1) / EV_TR);
        int rc = 0;
        if (ranges > 0) {
            EvalParams b = p;
            b.k = kp;
            b.splits = ranges;
            b.tiles_per_split = tpr;
#define WR_EVAL_LONG(DD) rc = launch_eval<DD, 3>(b, st, row_tiles); if (!rc) rc = launch_eval<DD, 2>(p, st, row_tiles)
            switch (D) {
                case 16: WR_EVAL_LONG(16); break;
                case 32: WR_EVAL_LONG(32); break;
                case 64: WR_EVAL_LONG(64); break;
                case 128: WR_EVAL_LONG(128); break;
                default: WR_EVAL_LONG(256); break;
            }
#undef WR_EVAL_LONG
        } else {
            switch (D) {
                case 16: rc = launch_eval<16, 2>(p, st, row_tiles); break;
                case 32: rc = launch_eval<32, 2>(p, st, row_tiles); break;
                case 64: rc = launch_eval<64, 2>(p, st, row_tiles); break;
                case 128: rc = launch_eval<128, 2>(p, st, row_tiles); break;
                default: rc = launch_eval<256, 2>(p, st, row_tiles); break;
            }
        }
        if (rc) return rc;
        LongSelect q{lg.seg, lg.seg_cnt, rn, p.Uemb, p.user, target_in ? 1 : 0, Iemb, D, n_items, hist_ptr, hist_idx, k,
                     topk_idx + r0 * k, topk_val + r0 * k, fallback, &((WrWorkspace *)ws)->status};
        rc = long_select(q, st);
        if (rc) return rc;
    }
    return WR_OK;
}

extern "C" int wr_eval_rank_topk_long(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos,
                                      int64_t R, int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr,
                                      const int32_t *hist_idx, int k, int precision, int32_t *topk_idx, float *topk_val,
                                      int32_t *rank, float *target, void *scratch, void *ws, void *stream) {
    if (!target) return WR_E_NULL;
    return eval_rank_topk_long_impl(Uemb, Iemb, user, pos, R, n_users, n_items, D, hist_ptr, hist_idx, k, precision,
                                    topk_idx, topk_val, rank, target, nullptr, scratch, ws, stream);
}

extern "C" int wr_eval_rank_topk_long_shard(const float *Urows, const float *Iemb, const int64_t *user,
                                            const int64_t *pos_local, int64_t R, int64_t n_users, int64_t n_items_local,
                                            int D, const int64_t *hist_ptr, const int32_t *hist_idx, int k,
                                            int precision, const float *target, int32_t *topk_idx, float *topk_val,
                                            int32_t *rank, void *scratch, void *ws, void *stream) {
    if (!target) return WR_E_NULL;
    return eval_rank_topk_long_impl(Urows, Iemb, user, pos_local, R, n_users, n_items_local, D, hist_ptr, hist_idx, k,
                                    precision, topk_idx, topk_val, rank, nullptr, target, scratch, ws, stream);
}

extern "C" int wr_metrics(const int32_t *rank, int64_t R, const int *host_ks, int nk, double *out, void *ws,
                          void *stream) {
    if (!rank || !host_ks || !out || !ws) return WR_E_NULL;
    if (R <= 0 || nk < 1 || nk > 8) return WR_E_SIZE;
    int ks[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < nk; ++i) ks[i] = host_ks[i];
    int64_t g = (R + 255) / 256;
    if (g > 64) g = 64;
    metrics_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(rank, R, nk, ks[0], ks[1], ks[2], ks[3], ks[4], ks[5],
                                                              ks[6], ks[7], out, (WrWorkspace *)ws);
    WR_CHECK_LAUNCH();
    return WR_OK;
}
