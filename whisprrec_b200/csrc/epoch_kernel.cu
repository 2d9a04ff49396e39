// The resident BPRMF training kernel: every step of BaseRunner.fit's loop (BaseRunner.py:194-200) inside ONE
// cooperative launch, for tables whose Adam state fits in the shared memory of the SMs (ml-100k / ml-1m sized).
//
//   * one CTA per SM; CTA c owns a contiguous 1/grid of the fused table: its P / M / V live in shared memory for
//     the whole launch (M and V never touch L2 between steps; P is published to global memory after every update
//     because the next step's gathers read it), G is the only array read and re-zeroed through L2;
//   * 16 worker warps: BPR phase (ids from shared memory -> 3 rows from L2 -> dots -> REDs into G), grid barrier,
//     Adam phase on the CTA's slice, grid barrier;
//   * one helper warp per CTA runs AHEAD of the workers: it stages the ids of the next steps into shared memory (so no
//     global or PCIe latency sits between the barrier and the first row gather) and, for the steps it is on duty for
//     (step % grid == CTA), sums the per-CTA loss partials in CTA order and delivers the loss -- off the workers'
//     critical path;
//   * streaming (host-fed) mode: one more warp in CTA 0 polls a descriptor ring in mapped host memory, forwards new
//     descriptors to a device ring and releases the steps; the helpers read the ids straight from pinned host memory
//     (the H2D transfer) and deliver loss + completion words to mapped host memory (the D2H transfer).  The kernel leaves
//     when the host closes the stream or has not fed it for `idle_ns`.
//
// Single steps (wr_bprmf_step) stay on the L2-streamed cooperative kernel of train_kernels.cu: with a cold L2 and one
// step per launch there is nothing for the shared-memory state to amortise (measured: 18.5 vs 14.3 us, scripts/prof_resident.py).
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"

namespace wr {

constexpr int EP_THREADS = 512;                 // worker threads
constexpr int EP_WARPS = EP_THREADS / 32;
constexpr int EP_BLOCK = EP_THREADS + 64;       // + helper warp + poller warp
constexpr int EP_STAGE_DEPTH = 4;               // steps the helper may run ahead of the workers
constexpr int EP_STAGE_CAP = 128;               // interactions per CTA and step: batch <= 128 x grid
constexpr int EP_PD = WR_EP_PART_DEPTH;
constexpr uint32_t EP_COUNT_MASK = 0x3fffffffu;
constexpr uint64_t EP_TIMEOUT_NS = 5000000000ull;   // a grid barrier that takes 5 s is a bug or a dead peer CTA

struct StepDesc {            // 32 bytes; `seq` is written last by the host (streaming mode)
    const int64_t *ids;      // user ids of the batch; positives at ids + stride, negatives at ids + 2 stride
    int64_t stride;
    int32_t B;               // rows; -1 closes the stream
    float step_size, bc2_sqrt;
    uint32_t seq;            // step + 1
};
static_assert(sizeof(StepDesc) == 32, "StepDesc is copied as eight 32-bit words");

struct Stage {
    int32_t u[EP_STAGE_CAP], i[EP_STAGE_CAP], j[EP_STAGE_CAP];
    int32_t B, mine;
    float step_size, bc2_sqrt;
};

struct EpochParams {
    float4 *P, *M, *V, *G;
    int64_t n4, chunk;                 // float4 per array; float4 per CTA
    int64_t n_users, n_items;
    float gamma, l2, w1, beta2, w2, eps;
    const StepDesc *desc;              // device ring
    uint32_t desc_ring;
    uint32_t first_step, preset_count; // not streaming: steps [first_step, preset_count) exist from the start
    float *losses;                     // device, losses[s - first_step] (nullable)
    WrWorkspace *ws;
    // streaming
    const StepDesc *host_desc;         // mapped host ring (nullptr = not streaming)
    uint32_t host_ring;
    uint32_t *host_lossq;              // [host_ring][2] {step + 1, loss bits} once the loss is out
    uint32_t *host_done;               // [host_ring] step + 1 once the step is complete
    uint32_t *host_exit;               // steps processed + 1 when the kernel leaves on its own (idle)
    uint64_t idle_ns;
    int64_t *dev_ids;                  // device ring [host_ring][3 * dev_ids_cap]: the helpers' copy of each step's ids
    int64_t dev_ids_cap;
    // owner-computes form (bprmf_epoch_owner_kernel): rows per CTA, ids per staged step, staged steps
    int32_t rows_per_cta, bcap, depth;
    uint64_t *trace;                   // profiling (wr_debug_epoch_trace): [step - first_step][8] globaltimer stamps
    uint64_t *cta_trace;               // profiling: [step - first_step][grid][4] arrival / passage of both barriers, every CTA
};

// trace slots: 0 step start, 1 BPR done, 2 past barrier 1, 3 Adam done, 4 past barrier 2 (CTA 0's thread 0);
// 5 descriptor seen by the poller, 6 ids staged by CTA 0's helper, 7 completion word written by the duty helper
__device__ __forceinline__ void trace_stamp(const EpochParams &p, uint32_t step, int slot) {
    if (p.trace) p.trace[(size_t)(step - p.first_step) * 8 + slot] = global_timer_ns();
}

__device__ __forceinline__ void workers_sync() { asm volatile("bar.sync 1, %0;" ::"n"(EP_THREADS) : "memory"); }

__device__ __forceinline__ uint32_t lds_acquire(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void sts_release(uint32_t *p, uint32_t v) {
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int64_t ld_relaxed_sys_s64(const int64_t *p) {
    int64_t v;
    asm volatile("ld.relaxed.sys.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem)
                 : "memory");
}

__device__ __forceinline__ uint4 ld_relaxed_sys_v4(const void *p) {
    uint4 v;
    asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}

// Grid barrier of the worker threads, number `value` (1, 2, 3, ... within a launch).  No counter: CTA c publishes its
// arrival number in its own 128-byte line and thread t of every CTA waits for CTA t's -- one store, one load round,
// no serialised atomics (148 atomics on one word cost ~0.6 us).  The caller has synchronised the workers.  `extra`
// (nullable) is one more word thread 0 waits for while it spins anyway: *extra >= extra_min.  Returns false when the
// wait was abandoned (timeout / another CTA gave up).
__device__ __forceinline__ bool grid_barrier(WrWorkspace *ws, uint32_t value, uint32_t *s_abort, const uint32_t *extra,
                                             uint32_t extra_min, bool arrive = true) {
    const int tid = threadIdx.x;
    if (arrive && tid == 0) st_release_gpu(&ws->ep_flag[32 * blockIdx.x], value);
    if (tid < (int)gridDim.x) {
        const uint32_t *f = &ws->ep_flag[32 * tid];
        uint64_t t0 = 0;
        uint32_t spins = 0;
        bool ok_extra = tid != 0 || extra == nullptr;
        for (;;) {
            if (!ok_extra) ok_extra = (int32_t)(ld_acquire_u32(extra) - extra_min) >= 0;
            if (ok_extra && (int32_t)(ld_acquire_u32(f) - value) >= 0) break;
            if ((++spins & 255u) == 0) {
                if (ld_acquire_u32(&ws->ep_abort)) { *s_abort = 1; break; }
                const uint64_t now = global_timer_ns();
                if (t0 == 0) t0 = now;
                if (now - t0 > EP_TIMEOUT_NS) {
                    atomicOr(&ws->status, WR_STATUS_PEER_TIMEOUT);
                    atomicExch(&ws->ep_abort, 1u);
                    *s_abort = 1;
                    break;
                }
            }
        }
    }
    workers_sync();
    return *(volatile uint32_t *)s_abort == 0;
}

// Helper warp: has every CTA arrived at barrier number `value`?
__device__ __forceinline__ bool all_arrived(const WrWorkspace *ws, uint32_t value) {
    bool ok = true;
    for (int i = threadIdx.x & 31; i < (int)gridDim.x; i += 32) ok = ok && (int32_t)(ld_acquire_u32(&ws->ep_flag[32 * i]) - value) >= 0;
    return __all_sync(0xffffffffu, ok);
}

// ---- the helper warp: stages ids ahead of the workers, reduces the loss of the steps it is on duty for ----
struct StageHdr {            // owner-computes form: the ids themselves live in dynamic shared memory, [depth][3][bcap] int64
    int32_t B;
    float step_size, bc2_sqrt;
};

template <bool OWNER>
__device__ void epoch_helper(const EpochParams &p, Stage *stage, uint32_t *s_ready, uint32_t *s_consumed,
                             uint32_t *s_exit_at, uint32_t *s_abort, int32_t *s_B, StageHdr *hdr = nullptr,
                             int64_t *stage_ids = nullptr) {
    const uint32_t stage_depth = OWNER ? (uint32_t)p.depth : (uint32_t)EP_STAGE_DEPTH;
    const int lane = threadIdx.x & 31, cta = blockIdx.x, grid = gridDim.x;
    const bool streaming = p.host_desc != nullptr;
    WrWorkspace *ws = p.ws;
    uint32_t n = p.first_step, nf = p.first_step;
    uint32_t duty = p.first_step + (uint32_t)((cta + grid - (int)(p.first_step % (uint32_t)grid)) % grid);
    int duty_state = 0;
    uint32_t count = streaming ? p.first_step : p.preset_count;
    bool closed = !streaming, exit_published = false;
    uint64_t t_idle = 0;
    for (;;) {
        bool progress = false;
        StepDesc fresh;
        bool have_fresh = false;
        if (streaming && !closed) {
            // the poller forwards descriptors into the device ring as single 32-byte stores: slot `count` is valid once its
            // seq word says so (no separate "go" word, no fence: descriptor and signal are the same sector)
            const uint4 *src = reinterpret_cast<const uint4 *>(p.desc + count % p.desc_ring);
            const uint4 a = __ldcg(src), b = __ldcg(src + 1);
            memcpy(&fresh, &a, 16);
            memcpy(reinterpret_cast<char *>(&fresh) + 16, &b, 16);
            if (fresh.seq == count + 1u) {
                if (fresh.B < 0) {
                    closed = true;
                } else {
                    have_fresh = nf == count;
                    ++count;
                }
                progress = true;
            }
        }
        // ---- loss duty (first: its partial slot gates the workers four steps later) ----
        if (duty < n) {
            const uint32_t rel = duty - p.first_step;
            if (duty_state == 0) {
                if (all_arrived(ws, OWNER ? rel + 1u : 2u * rel + 1u)) {
                    float t = 0.f;
                    for (int i = lane; i < grid; i += 32) t += __ldcg(&ws->ep_partial[(duty % EP_PD) * WR_EP_MAX_GRID + i]);
                    t = warp_sum(t);
                    if (lane == 0) {
                        const float loss = t / (float)s_B[duty % EP_PD];
                        if (p.losses) p.losses[rel] = loss;
                        if (streaming)      // loss and its sequence word travel as ONE 8-byte store: no sys-scope fence (a PCIe round trip)
                            asm volatile("st.relaxed.sys.global.v2.b32 [%0], {%1, %2};" ::"l"(p.host_lossq + 2 * (duty % p.host_ring)),
                                         "r"(duty + 1u), "r"(__float_as_uint(loss)) : "memory");
                        st_release_gpu(&ws->ep_loss_flag[duty % EP_PD], duty + 1u);
                    }
                    duty_state = streaming ? 1 : 2;
                    progress = true;
                }
            }
            if (duty_state == 1) {      // streaming: the step is complete once every CTA is through its second barrier
                if (all_arrived(ws, OWNER ? rel + 1u : 2u * rel + 2u)) {
                    if (lane == 0) {
                        // every CTA's P stores were released at gpu scope before its arrival, which this warp has acquired
                        asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p.host_done + duty % p.host_ring), "r"(duty + 1u) : "memory");
                        trace_stamp(p, duty, 7);
                    }
                    duty_state = 2;
                    progress = true;
                }
            }
            if (duty_state == 2) {
                duty += (uint32_t)grid;
                duty_state = 0;
            }
        }
        // ---- streaming: copy this helper's piece of step nf's ids out of pinned host memory into the device ring
        //      (16-byte loads, every helper a contiguous 128-byte-aligned piece: a few hundred PCIe reads per step
        //      instead of one per id) ----
        if (streaming && nf < count && nf - lds_acquire(s_consumed) < stage_depth + 2u) {
            StepDesc d = fresh;
            if (!have_fresh) {
                const uint4 *src = reinterpret_cast<const uint4 *>(p.desc + nf % p.desc_ring);
                const uint4 a = __ldcg(src), b = __ldcg(src + 1);
                memcpy(&d, &a, 16);
                memcpy(reinterpret_cast<char *>(&d) + 16, &b, 16);
            }
            const int total16 = (3 * d.B + 1) >> 1;                         // 16-byte units of the [3, B] int64 block
            const int per16 = (((total16 + grid - 1) / grid) + 7) & ~7;
            const int lo = cta * per16, hi = min(total16, lo + per16);
            const uint4 *hsrc = reinterpret_cast<const uint4 *>(d.ids);
            uint4 *ddst = reinterpret_cast<uint4 *>(p.dev_ids + (size_t)(nf % p.host_ring) * 3 * p.dev_ids_cap);
            for (int k = lo + lane; k < hi; k += 32) __stcg(ddst + k, ld_relaxed_sys_v4(hsrc + k));
            __syncwarp();
            if (lane == 0) {
                __threadfence();
                atomicAdd(&ws->ep_fetched[(nf - p.first_step) & 15u], 1u);
            }
            ++nf;
            progress = true;
        }
        // ---- stage the ids of step n ----
        bool can_stage = n < count && !(duty < n && n >= duty + EP_PD);       // s_B[duty % EP_PD] must outlive the duty
        if (can_stage && streaming) {
            can_stage = n < nf;
            if (can_stage) {
                const uint32_t reln = n - p.first_step;
                uint32_t f = lane == 0 ? ld_acquire_u32(&ws->ep_fetched[reln & 15u]) : 0u;
                f = __shfl_sync(0xffffffffu, f, 0);
                can_stage = (int32_t)(f - ((reln >> 4) + 1u) * (uint32_t)grid) >= 0;
            }
        }
        if (can_stage) {
            const uint32_t cons = lds_acquire(s_consumed);
            if (n - cons < stage_depth) {
                StepDesc d;
                {
                    const uint4 *src = reinterpret_cast<const uint4 *>(p.desc + n % p.desc_ring);
                    const uint4 a = __ldcg(src), b = __ldcg(src + 1);
                    memcpy(&d, &a, 16);
                    memcpy(reinterpret_cast<char *>(&d) + 16, &b, 16);
                }
                if (streaming) {       // the device copy: [3, B] packed
                    d.ids = p.dev_ids + (size_t)(n % p.host_ring) * 3 * p.dev_ids_cap;
                    d.stride = d.B;
                }
                const int B = d.B;
                if (OWNER) {
                    // every id of the step goes into shared memory as it is (8-byte async copies, all in flight at once:
                    // a converting loop on one warp is a chain of L2 round trips -- measured 13 us per step)
                    int64_t *su = stage_ids + (size_t)(n % stage_depth) * 3 * p.bcap;
                    if (streaming) {
                        // the device ring is rewritten while the kernel runs: L2 only (.cg, 16 bytes), the packed [3 B] block
                        const int total16 = (3 * B + 1) >> 1;
                        const uint4 *src = reinterpret_cast<const uint4 *>(d.ids);
                        uint4 *dst = reinterpret_cast<uint4 *>(su);
                        for (int k = lane; k < total16; k += 32) cp_async16(dst + k, src + k);
                    } else {
                        for (int r = 0; r < 3; ++r) {      // ids that exist before the launch; any 8-byte alignment
                            const int64_t *src = d.ids + r * d.stride;
                            int64_t *dst = su + (size_t)r * B;
                            for (int b = lane; b < B; b += 32)
                                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst + b)),
                                             "l"(src + b) : "memory");
                        }
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    asm volatile("cp.async.wait_all;" ::: "memory");
                    if (lane == 0) {
                        StageHdr &h = hdr[n % stage_depth];
                        h.B = B;
                        h.step_size = d.step_size;
                        h.bc2_sqrt = d.bc2_sqrt;
                        s_B[n % EP_PD] = B;
                    }
                    __syncwarp();
                    if (lane == 0 && cta == 0) trace_stamp(p, n, 6);
                    if (lane == 0) sts_release(s_ready, n + 1u);
                    ++n;
                    progress = true;
                    continue;
                }
                const int per = (B + grid - 1) / grid;
                int mine = B - cta * per;
                mine = mine < 0 ? 0 : (mine > per ? per : mine);
                Stage &st = stage[n % EP_STAGE_DEPTH];
                for (int q = lane; q < mine; q += 32) {
                    const int64_t b = (int64_t)cta * per + q;
                    const int64_t u = __ldcg(d.ids + b), i = __ldcg(d.ids + d.stride + b), j = __ldcg(d.ids + 2 * d.stride + b);
                    const bool ok = (uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
                                    (uint64_t)j < (uint64_t)p.n_items;
                    if (!ok) atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
                    st.u[q] = ok ? (int32_t)u : -1;
                    st.i[q] = ok ? (int32_t)i : -1;
                    st.j[q] = ok ? (int32_t)j : -1;
                }
                if (lane == 0) {
                    st.B = B;
                    st.mine = mine;
                    st.step_size = d.step_size;
                    st.bc2_sqrt = d.bc2_sqrt;
                    s_B[n % EP_PD] = B;
                }
                __syncwarp();
                if (lane == 0 && cta == 0) trace_stamp(p, n, 6);
                if (lane == 0) sts_release(s_ready, n + 1u);
                ++n;
                progress = true;
            }
        }
        if (closed && n >= count) {
            if (!exit_published) {
                if (lane == 0) sts_release(s_exit_at, count);
                exit_published = true;
            }
            if (duty >= count) break;
        }
        if (progress) {
            t_idle = 0;
            continue;
        }
        // nothing to do right now: look for an abandoned launch, then yield the issue slots to the workers
        uint32_t ab = lane == 0 ? (ld_acquire_u32(&ws->ep_abort) | *(volatile uint32_t *)s_abort) : 0u;
        ab = __shfl_sync(0xffffffffu, ab, 0);
        if (ab) break;
        if (!streaming) {       // a step that never completes (the streaming kernel idles legitimately; its poller decides)
            const uint64_t now = global_timer_ns();
            if (t_idle == 0) t_idle = now;
            if (now - t_idle > 2 * EP_TIMEOUT_NS) {
                if (lane == 0) {
                    atomicOr(&ws->status, WR_STATUS_PEER_TIMEOUT);
                    atomicExch(&ws->ep_abort, 1u);
                }
                break;
            }
        }
        __nanosleep(40);
    }
}

// ---- the poller warp (CTA 0, streaming): host descriptor ring -> device ring (which releases the step) ----
__device__ void epoch_poller(const EpochParams &p) {
    const int lane = threadIdx.x & 31;
    WrWorkspace *ws = p.ws;
    uint32_t forwarded = p.first_step;
    uint64_t t_act = global_timer_ns();
    for (;;) {
        // one 32-byte read over PCIe: the descriptor of the next step, valid once its seq word (written last) matches
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.host_desc + forwarded % p.host_ring);
        uint32_t w = lane < 8 ? ld_relaxed_sys_u32(src + lane) : 0u;
        const uint32_t seq = __shfl_sync(0xffffffffu, w, 7);
        const int32_t B = (int32_t)__shfl_sync(0xffffffffu, w, 4);
        const uint64_t now = global_timer_ns();
        uint32_t *dst = reinterpret_cast<uint32_t *>(const_cast<StepDesc *>(p.desc) + forwarded % p.desc_ring);
        if (seq == forwarded + 1u) {
            if (lane < 8) __stcg(dst + lane, w);      // one 32-byte sector: the helpers see all of it or none
            if (B < 0) break;                         // the host closed the stream after `forwarded` steps
            if (lane == 0) trace_stamp(p, forwarded, 5);
            ++forwarded;
            t_act = now;
            continue;
        }
        if (ld_acquire_u32(&ws->ep_abort)) break;
        if (now - t_act > p.idle_ns) {                // not fed for a while: close the stream ourselves and tell the host
            if (lane < 8) __stcg(dst + lane, lane == 4 ? 0xffffffffu : (lane == 7 ? forwarded + 1u : 0u));
            if (lane == 0) st_release_sys(p.host_exit, forwarded + 1u);
            break;
        }
    }
}

// Every party that touches the control words (workers and helper of every CTA, the poller) checks out here; the last
// one re-arms the words for the next launch.
__device__ __forceinline__ void epoch_depart(const EpochParams &p) {
    WrWorkspace *ws = p.ws;
    __threadfence();
    const uint32_t parties = 2u * gridDim.x + (p.host_desc ? 1u : 0u);
    const uint32_t t = atomicAdd(&ws->ep_depart, 1u);
    if (t == parties - 1u) {
        for (int i = 0; i < 16; ++i) ws->ep_fetched[i] = 0;
        for (int i = 0; i < (int)gridDim.x; ++i) ws->ep_flag[32 * i] = 0;
        ws->ep_abort = 0;
        for (int i = 0; i < EP_PD; ++i) ws->ep_loss_flag[i] = 0;
        __threadfence();
        ws->ep_depart = 0;
    }
}

template <int LPR, int VPL>
__global__ void __maxnreg__(64) bprmf_epoch_kernel(const EpochParams p) {
    using RG = RowGroup<LPR, VPL>;
    constexpr int D = RG::D, GROUPS = RG::GROUPS;
    extern __shared__ float4 smem4[];
    __shared__ Stage stage[EP_STAGE_DEPTH];
    __shared__ uint32_t s_ready, s_consumed, s_exit_at, s_abort, s_run;
    __shared__ int32_t s_B[EP_PD];
    __shared__ float s_red[EP_WARPS];
    const int tid = threadIdx.x, cta = blockIdx.x, grid = gridDim.x;
    WrWorkspace *ws = p.ws;
    if (tid == 0) {
        s_ready = p.first_step;
        s_consumed = p.first_step;
        s_exit_at = 0xffffffffu;
        s_abort = 0;
        s_run = 0;
    }
    __syncthreads();
    if (tid >= EP_THREADS) {
        const bool helper = tid < EP_THREADS + 32;
        if (helper) {
            epoch_helper<false>(p, stage, &s_ready, &s_consumed, &s_exit_at, &s_abort, s_B);
            if ((tid & 31) == 0) epoch_depart(p);
        } else if (cta == 0 && p.host_desc) {
            epoch_poller(p);
            if ((tid & 31) == 0) epoch_depart(p);
        }
        return;
    }
    // =========================== workers ===========================
    const int64_t lo4 = (int64_t)cta * p.chunk;
    int cnt = (int)(p.n4 - lo4 < p.chunk ? p.n4 - lo4 : p.chunk);
    if (cnt < 0) cnt = 0;
    float4 *sP = smem4, *sM = sP + p.chunk, *sV = sM + p.chunk;
    float4 *gP = p.P + lo4, *gM = p.M + lo4, *gV = p.V + lo4, *gG = p.G + lo4;
    // phase 0: the CTA's slice of P / M / V streams into shared memory behind the first step's BPR phase
    for (int k = tid; k < cnt; k += EP_THREADS) {
        cp_async16(sP + k, gP + k);
        cp_async16(sM + k, gM + k);
        cp_async16(sV + k, gV + k);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (tid == 32 && cnt > 0)       // cold L2 (first step after other work): the gradient slice is on its way before the REDs
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gG), "r"((uint32_t)cnt * 16u) : "memory");
    const int lane = tid & 31, sub = lane % LPR, grp = lane / LPR, warp = tid >> 5;
    const float *Ub = reinterpret_cast<const float *>(p.P), *Ib = Ub + p.n_users * D;
    float *gUb = reinterpret_cast<float *>(p.G), *gIb = gUb + p.n_users * D;
    const bool streaming = p.host_desc != nullptr;
    bool loaded = false, aborted = false;
    uint32_t s = p.first_step;
    for (;; ++s) {
        if (tid == 0) {
            uint32_t run = 1;
            for (uint32_t spins = 0;; ++spins) {
                if ((int32_t)(lds_acquire(&s_ready) - (s + 1u)) >= 0) break;
                if (lds_acquire(&s_exit_at) <= s) { run = 0; break; }
                if ((spins & 1023u) == 1023u && (ld_acquire_u32(&ws->ep_abort) | *(volatile uint32_t *)&s_abort)) { run = 0; s_abort = 1; break; }
            }
            s_run = run;
        }
        workers_sync();
        if (!*(volatile uint32_t *)&s_run) break;
        const uint32_t rel = s - p.first_step;
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 0);
        const Stage &st = stage[s % EP_STAGE_DEPTH];
        const int mine = st.mine;
        const float coef = 1.0f / (float)st.B;
        AdamScalars sc{p.l2, p.w1, p.beta2, p.w2, p.eps, st.step_size, st.bc2_sqrt};
        const float inv_bc2 = 1.0f / st.bc2_sqrt;
        // ---- BPR forward + backward on this CTA's rows of the batch ----
        float local = 0.f;
        for (int q0 = warp * GROUPS; q0 < mine; q0 += EP_WARPS * GROUPS) {
            const int q = q0 + grp;
            int u = -1, i = -1, j = -1;
            if (q < mine) {
                u = st.u[q];
                i = st.i[q];
                j = st.j[q];
            }
            const bool ok = u >= 0;
            float4 ue[VPL], pe[VPL], ne[VPL];
            if (ok) {
                RG::load_cg(Ub + (int64_t)u * D, sub, ue);
                RG::load_cg(Ib + (int64_t)i * D, sub, pe);
                RG::load_cg(Ib + (int64_t)j * D, sub, ne);
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
                bpr_pointwise(sp, sn, p.gamma, coef, l, c);
                if (sub == 0) local += l;
                float *gu = gUb + (int64_t)u * D, *gp = gIb + (int64_t)i * D, *gn = gIb + (int64_t)j * D;
#pragma unroll
                for (int v = 0; v < VPL; ++v) {
                    const int off = 4 * (sub + v * LPR);
                    red_add_v4(gu + off, scale4(sub4(pe[v], ne[v]), c));
                    red_add_v4(gp + off, scale4(ue[v], c));
                    red_add_v4(gn + off, scale4(ue[v], -c));
                }
            }
        }
        local = warp_sum(local);
        if (lane == 0) s_red[warp] = local;
        if (!loaded) asm volatile("cp.async.wait_all;" ::: "memory");
        workers_sync();
        loaded = true;
        if (tid == 0) {
            if (p.trace && cta == 0) trace_stamp(p, s, 1);
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < EP_WARPS; ++w) t += s_red[w];
            __stcg(&ws->ep_partial[(s % EP_PD) * WR_EP_MAX_GRID + cta], t);
            sts_release(&s_consumed, s + 1u);          // every worker has read its ids: the stage slot may be refilled
        }
        // ---- grid barrier 1: every gradient RED of the step has been performed ----
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 0] = global_timer_ns();
        if (!grid_barrier(ws, 2u * rel + 1u, &s_abort, nullptr, 0)) { aborted = true; break; }
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 1] = global_timer_ns();
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 2);
        // ---- Adam + L2 on the CTA's slice: state in shared memory, gradient from L2, P published, G re-zeroed ----
        const float4 z = f4_zero();
        for (int k = tid; k < cnt; k += 2 * EP_THREADS) {
            const int k2 = k + EP_THREADS;
            const bool two = k2 < cnt;
            float4 ga = __ldcg(gG + k), gb = z;
            if (two) gb = __ldcg(gG + k2);
            float4 pa = sP[k], ma = sM[k], va = sV[k];
            adam_elem_nr(pa.x, ma.x, va.x, ga.x, sc, inv_bc2);
            adam_elem_nr(pa.y, ma.y, va.y, ga.y, sc, inv_bc2);
            adam_elem_nr(pa.z, ma.z, va.z, ga.z, sc, inv_bc2);
            adam_elem_nr(pa.w, ma.w, va.w, ga.w, sc, inv_bc2);
            gP[k] = pa;
            gG[k] = z;
            sP[k] = pa;
            sM[k] = ma;
            sV[k] = va;
            if (two) {
                float4 pb = sP[k2], mb = sM[k2], vb = sV[k2];
                adam_elem_nr(pb.x, mb.x, vb.x, gb.x, sc, inv_bc2);
                adam_elem_nr(pb.y, mb.y, vb.y, gb.y, sc, inv_bc2);
                adam_elem_nr(pb.z, mb.z, vb.z, gb.z, sc, inv_bc2);
                adam_elem_nr(pb.w, mb.w, vb.w, gb.w, sc, inv_bc2);
                gP[k2] = pb;
                gG[k2] = z;
                sP[k2] = pb;
                sM[k2] = mb;
                sV[k2] = vb;
            }
        }
        // ---- grid barrier 2: every row of P is final, G is zero.  Not needed after the last step of a launch whose
        //      length is known up front; while it spins, thread 0 also waits for the loss of step s + 1 - EP_PD to
        //      have left the partial slot step s + 1 writes ----
        if (!streaming && s + 1u == p.preset_count) { ++s; break; }
        workers_sync();
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 3);
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 2] = global_timer_ns();
        const uint32_t nxt = s + 1u;
        const bool gate = nxt - p.first_step >= (uint32_t)EP_PD;
        if (!grid_barrier(ws, 2u * rel + 2u, &s_abort, gate ? &ws->ep_loss_flag[nxt % EP_PD] : nullptr,
                          nxt - (uint32_t)EP_PD + 1u)) { aborted = true; break; }
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 4);
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 3] = global_timer_ns();
    }
    // ---- leave: M and V go back to global memory (P is already there) ----
    if (loaded && !aborted) {
        for (int k = tid; k < cnt; k += EP_THREADS) {
            gM[k] = sM[k];
            gV[k] = sV[k];
        }
    } else if (!loaded) {
        asm volatile("cp.async.wait_all;" ::: "memory");
    }
    workers_sync();
    if (tid == 0) epoch_depart(p);
}

// ---- the owner-computes form: ONE grid barrier per step ---------------------------------------------------------------
// The two-barrier kernel above scatters gradient rows with REDs through L2, so Adam has to wait for every CTA's REDs
// (barrier 1) and the next step's gathers for every CTA's Adam (barrier 2).  Here the CTA that OWNS a row computes that
// row's gradient itself: every CTA scans the whole batch (ids staged in shared memory by its helper), keeps the
// (entry, role) pairs whose row it owns, evaluates those entries -- its own rows come from shared memory, the others
// from L2 -- and accumulates into a gradient slice that also lives in shared memory.  Nothing is exchanged between the
// BPR and the Adam phase any more.  What remains is the write-after-read hazard on P (a fast CTA's Adam must not
// overwrite rows a slow CTA is still gathering for the same step): the published copy of P is double-buffered in global
// memory -- step k reads buffer k & 1 and writes the other; the second buffer is G, which this kernel does not use
// otherwise and hands back zeroed -- so the only meeting point of a step is "the new P is complete".
//   * ownership is cyclic (row r belongs to CTA r % grid, local row r / grid): users, items and hot rows spread evenly;
//   * each batch entry is evaluated by up to three CTAs (the arithmetic is ~1 % of a step);
//   * the next step's ownership scan runs between a CTA's arrival at the barrier and its wait (ids and ownership only).
// x added into a float4 in shared memory.  There is no native fp32 add on shared memory (atomicAdd(float) compiles to one
// compare-and-swap loop per float); one 128-bit CAS covers the whole float4.
__device__ __forceinline__ void smem_add_f4(float4 *addr, float4 x) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(addr);
    float4 old = *addr;
    for (;;) {
        const float4 neu = make_float4(old.x + x.x, old.y + x.y, old.z + x.z, old.w + x.w);
        unsigned __int128 cmp, val, got;
        cmp = ((unsigned __int128)__float_as_uint(old.w) << 96) | ((unsigned __int128)__float_as_uint(old.z) << 64) |
              ((unsigned __int128)__float_as_uint(old.y) << 32) | (unsigned __int128)__float_as_uint(old.x);
        val = ((unsigned __int128)__float_as_uint(neu.w) << 96) | ((unsigned __int128)__float_as_uint(neu.z) << 64) |
              ((unsigned __int128)__float_as_uint(neu.y) << 32) | (unsigned __int128)__float_as_uint(neu.x);
        asm volatile("atom.shared.cas.b128 %0, [%1], %2, %3;" : "=q"(got) : "r"(a), "q"(cmp), "q"(val) : "memory");
        if (got == cmp) break;
        old.x = __uint_as_float((uint32_t)got);
        old.y = __uint_as_float((uint32_t)(got >> 32));
        old.z = __uint_as_float((uint32_t)(got >> 64));
        old.w = __uint_as_float((uint32_t)(got >> 96));
    }
}

__device__ __forceinline__ void grid_arrive(WrWorkspace *ws, uint32_t value) {
    if (threadIdx.x == 0) st_release_gpu(&ws->ep_flag[32 * blockIdx.x], value);
}

template <int LPR, int VPL>
__global__ void __maxnreg__(64) bprmf_epoch_owner_kernel(const EpochParams p) {
    using RG = RowGroup<LPR, VPL>;
    constexpr int D = RG::D, D4 = D / 4, GROUPS = RG::GROUPS, NG = EP_WARPS * GROUPS;
    extern __shared__ float4 smem4[];
    __shared__ StageHdr hdr[EP_STAGE_DEPTH];
    __shared__ uint32_t s_ready, s_consumed, s_exit_at, s_abort, s_run, s_next_ok;
    __shared__ uint32_t s_cnt[2];
    __shared__ int32_t s_B[EP_PD];
    __shared__ float s_red[EP_WARPS];
    const int tid = threadIdx.x, cta = blockIdx.x, grid = gridDim.x;
    WrWorkspace *ws = p.ws;
    const int n_rows = (int)(p.n_users + p.n_items);
    const int my_rows = n_rows > cta ? (n_rows - cta + grid - 1) / grid : 0;       // rows cta, cta + grid, ...
    const int cnt = my_rows * D4;
    // r / grid for r < 2^24 by one 64-bit multiply (exact: the error term r / 2^40 stays below 1 / grid)
    const uint64_t magic = ((1ull << 40) + (uint64_t)grid - 1) / (uint64_t)grid;
    auto local_of = [&](int r, int &q) -> bool {         // does this CTA own row r?  q = its local row
        q = (int)(((uint64_t)(uint32_t)r * magic) >> 40);
        return r - q * grid == cta;
    };
    float4 *sP = smem4, *sM = sP + p.chunk, *sV = sM + p.chunk, *sG = sV + p.chunk;
    int64_t *stage_ids = reinterpret_cast<int64_t *>(sG + p.chunk);                 // [depth][3 bcap], a step's [3][B] packed
    int32_t *lists = reinterpret_cast<int32_t *>(stage_ids + (size_t)p.depth * 3 * p.bcap);   // [2][3 bcap]
    if (tid == 0) {
        s_ready = p.first_step;
        s_consumed = p.first_step;
        s_exit_at = 0xffffffffu;
        s_abort = 0;
        s_run = 0;
        s_next_ok = 0;
        s_cnt[0] = 0;
        s_cnt[1] = 0;
    }
    __syncthreads();
    if (tid >= EP_THREADS) {
        const bool helper = tid < EP_THREADS + 32;
        if (helper) {
            epoch_helper<true>(p, nullptr, &s_ready, &s_consumed, &s_exit_at, &s_abort, s_B, hdr, stage_ids);
            if ((tid & 31) == 0) epoch_depart(p);
        } else if (cta == 0 && p.host_desc) {
            epoch_poller(p);
            if ((tid & 31) == 0) epoch_depart(p);
        }
        return;
    }
    // =========================== workers ===========================
    // global float4 index of element k of the slice: local row k / D4 is global row (k / D4) * grid + cta
    auto gidx = [&](int k) -> int64_t { return ((int64_t)(k / D4) * grid + cta) * D4 + (k % D4); };
    for (int k = tid; k < cnt; k += EP_THREADS) {
        const int64_t g = gidx(k);
        cp_async16(sP + k, p.P + g);
        cp_async16(sM + k, p.M + g);
        cp_async16(sV + k, p.V + g);
        sG[k] = f4_zero();
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int lane = tid & 31, sub = lane % LPR, grp = lane / LPR, warp = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    float *sGf = reinterpret_cast<float *>(sG);
    const int n_users = (int)p.n_users;

    // Which (entry, role) pairs of step `step` touch a row this CTA owns -> lists[step & 1], s_cnt[step & 1].
    // Ids outside their table drop the whole entry (CTA 0 reports them).
    // Warps [w0, EP_WARPS) take part (the look-ahead scan leaves the first warps to poll the barrier flags meanwhile).
    auto scan = [&](uint32_t step, int w0) {
        if (warp < w0) return;
        const int B = hdr[step % (uint32_t)p.depth].B;
        const int64_t *su = stage_ids + (size_t)(step % (uint32_t)p.depth) * 3 * p.bcap, *si = su + B, *sj = si + B;
        int32_t *list = lists + (size_t)(step & 1u) * 3 * p.bcap;
        uint32_t *count = &s_cnt[step & 1u];
        // no warp-collective compaction: a lane that finds one of its rows here takes a slot with a shared-memory atomic
        // (a CTA owns 1 / grid of the rows: ~3 B / grid hits per step, and most warps see none in an iteration)
#pragma unroll 2
        for (int b = (warp - w0) * 32 + lane; b < B; b += (EP_WARPS - w0) * 32) {
            const int64_t u = su[b], i = si[b], j = sj[b];
            const bool valid = (uint64_t)u < (uint64_t)p.n_users && (uint64_t)i < (uint64_t)p.n_items &&
                               (uint64_t)j < (uint64_t)p.n_items;
            if (!valid) {
                if (cta == 0) atomicOr(&ws->status, WR_STATUS_INDEX_OUT_OF_RANGE);
                continue;
            }
            int q;
            if (local_of((int)u, q)) list[atomicAdd(count, 1u)] = (b << 2) | 0;
            if (local_of(n_users + (int)i, q)) list[atomicAdd(count, 1u)] = (b << 2) | 1;
            if (local_of(n_users + (int)j, q)) list[atomicAdd(count, 1u)] = (b << 2) | 2;
        }
    };

    bool loaded = false, aborted = false, scanned = false;
    uint32_t s = p.first_step;
    for (;; ++s) {
        if (!scanned) {      // (a step that was scanned ahead is known to be staged: straight on from the barrier)
            if (tid == 0) {
                uint32_t run = 1;
                for (uint32_t spins = 0;; ++spins) {
                    if ((int32_t)(lds_acquire(&s_ready) - (s + 1u)) >= 0) break;
                    if (lds_acquire(&s_exit_at) <= s) { run = 0; break; }
                    if ((spins & 1023u) == 1023u && (ld_acquire_u32(&ws->ep_abort) | *(volatile uint32_t *)&s_abort)) { run = 0; s_abort = 1; break; }
                }
                s_run = run;
            }
            if (!loaded) asm volatile("cp.async.wait_all;" ::: "memory");
            workers_sync();
            loaded = true;
            if (!*(volatile uint32_t *)&s_run) break;
        }
        const uint32_t rel = s - p.first_step;
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 0);
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 0] = global_timer_ns() | (scanned ? 0ull : 1ull);
        if (!scanned) {              // the previous step could not look ahead (first step / ids not staged in time)
            scan(s, 0);
            workers_sync();
        }
        const StageHdr h = hdr[s % (uint32_t)p.depth];
        const int64_t *su = stage_ids + (size_t)(s % (uint32_t)p.depth) * 3 * p.bcap, *si = su + h.B, *sj = si + h.B;
        const int32_t *list = lists + (size_t)(s & 1u) * 3 * p.bcap;
        const int L = (int)*(volatile uint32_t *)&s_cnt[s & 1u];
        const float coef = 1.0f / (float)h.B;
        AdamScalars sc{p.l2, p.w1, p.beta2, p.w2, p.eps, h.step_size, h.bc2_sqrt};
        const float inv_bc2 = 1.0f / h.bc2_sqrt;
        // the published copy of P this step gathers from, and the one its Adam writes
        const float4 *Rd = (rel & 1u) ? p.G : p.P;
        float4 *Wr = (rel & 1u) ? p.P : p.G;
        // ---- BPR forward + backward for those entries; the gradient of OUR row goes into the shared-memory slice ----
        float local = 0.f;
        for (int e0 = warp * GROUPS; e0 < L; e0 += NG) {
            const int e = e0 + grp;
            const bool ok = e < L;
            int role = 0, ru = 0, rp = 0, rn = 0;
            if (ok) {
                const int ent = list[e];
                const int b = ent >> 2;
                role = ent & 3;
                ru = (int)su[b];
                rp = n_users + (int)si[b];
                rn = n_users + (int)sj[b];
            }
            float4 ue[VPL], pe[VPL], ne[VPL];
            int mine_local = 0;
            if (ok) {
                int qu, qp, qn;
                const bool lu = local_of(ru, qu), lp = local_of(rp, qp), ln = local_of(rn, qn);
                mine_local = role == 0 ? qu : (role == 1 ? qp : qn);
#pragma unroll
                for (int v = 0; v < VPL; ++v) {
                    const int o = sub + v * LPR;
                    ue[v] = lu ? sP[qu * D4 + o] : __ldcg(Rd + (int64_t)ru * D4 + o);
                    pe[v] = lp ? sP[qp * D4 + o] : __ldcg(Rd + (int64_t)rp * D4 + o);
                    ne[v] = ln ? sP[qn * D4 + o] : __ldcg(Rd + (int64_t)rn * D4 + o);
                }
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
                bpr_pointwise(sp, sn, p.gamma, coef, l, c);
                if (role == 0 && sub == 0) local += l;
                float *g = sGf + (size_t)mine_local * D;
#pragma unroll
                for (int v = 0; v < VPL; ++v) {
                    const float4 x = role == 0 ? scale4(sub4(pe[v], ne[v]), c) : scale4(ue[v], role == 1 ? c : -c);
                    smem_add_f4(reinterpret_cast<float4 *>(g + 4 * (sub + v * LPR)), x);
                }
            }
        }
        local = warp_sum(local);
        if (lane == 0) s_red[warp] = local;
        workers_sync();
        if (tid == 0) {
            if (p.cta_trace) p.cta_trace[((size_t)rel * grid + cta) * 4 + 1] = global_timer_ns();
            if (p.trace && cta == 0) {
                trace_stamp(p, s, 1);
                trace_stamp(p, s, 2);          // (no barrier between the phases: slot 2 = slot 1)
            }
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < EP_WARPS; ++w) t += s_red[w];
            __stcg(&ws->ep_partial[(s % EP_PD) * WR_EP_MAX_GRID + cta], t);
            s_cnt[s & 1u] = 0;
            sts_release(&s_consumed, s + 1u);          // the ids of this step are no longer needed: the slot may be refilled
            // can the next step's scan run behind this step's arrival?  (its ids must be staged already)
            s_next_ok = (int32_t)(lds_acquire(&s_ready) - (s + 2u)) >= 0 ? 1u : 0u;
        }
        // ---- Adam + L2 on the slice: everything in shared memory; the new P goes to the OTHER published copy ----
        const float4 z = f4_zero();
        for (int k = tid; k < cnt; k += EP_THREADS) {
            float4 ga = sG[k], pa = sP[k], ma = sM[k], va = sV[k];
            adam_elem_nr(pa.x, ma.x, va.x, ga.x, sc, inv_bc2);
            adam_elem_nr(pa.y, ma.y, va.y, ga.y, sc, inv_bc2);
            adam_elem_nr(pa.z, ma.z, va.z, ga.z, sc, inv_bc2);
            adam_elem_nr(pa.w, ma.w, va.w, ga.w, sc, inv_bc2);
            Wr[gidx(k)] = pa;
            sP[k] = pa;
            sM[k] = ma;
            sV[k] = va;
            sG[k] = z;
        }
        workers_sync();
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 3);
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 2] = global_timer_ns();
        // ---- the step's only grid barrier: the new copy of P is complete (and the loss partials are out).  The arrival
        //      is published first; while it travels, the workers already pick the next step's entries.  While thread 0
        //      spins it also waits for the loss of step s + 1 - EP_PD to have left the partial slot step s + 1 writes.
        //      (The last step of a launch waits too: the clean-up below rewrites both copies.) ----
        grid_arrive(ws, rel + 1u);
        scanned = *(volatile uint32_t *)&s_next_ok != 0;
        const int poll_warps = (grid + 31) >> 5;        // the threads that watch the other CTAs' flags (grid_barrier)
        if (scanned) scan(s + 1u, poll_warps <= EP_WARPS - 4 ? poll_warps : 0);
        const uint32_t nxt = s + 1u;
        const bool gate = nxt - p.first_step >= (uint32_t)EP_PD;
        if (!grid_barrier(ws, rel + 1u, &s_abort, gate ? &ws->ep_loss_flag[nxt % EP_PD] : nullptr,
                          nxt - (uint32_t)EP_PD + 1u, false)) { aborted = true; break; }
        if (p.trace && cta == 0 && tid == 0) trace_stamp(p, s, 4);
        if (p.cta_trace && tid == 0) p.cta_trace[((size_t)rel * grid + cta) * 4 + 3] = global_timer_ns();
    }
    // ---- leave (every CTA is past the last step's barrier: nobody gathers any more): P, M and V of the slice go back to
    //      their tables, the slice of G -- the second published copy of P -- goes back to zero ----
    if (loaded && !aborted) {
        const float4 z = f4_zero();
        for (int k = tid; k < cnt; k += EP_THREADS) {
            const int64_t g = gidx(k);
            p.P[g] = sP[k];
            p.M[g] = sM[k];
            p.V[g] = sV[k];
            p.G[g] = z;
        }
    } else if (!loaded) {
        asm volatile("cp.async.wait_all;" ::: "memory");
    }
    workers_sync();
    if (tid == 0) epoch_depart(p);
}

// ---- host side ----------------------------------------------------------------------------------------------------
struct EpochConfig {
    int grid;
    int64_t chunk;
    size_t smem;
    const void *fn;
    int owner;                 // the one-barrier (owner-computes) kernel
    int rows_per_cta, bcap, depth;
};

template <int LPR, int VPL>
static int epoch_config_for(int64_t n4, EpochConfig *out) {
    static int sms = 0, max_smem = 0, attr_set = 0;
    const void *fn = (const void *)bprmf_epoch_kernel<LPR, VPL>;
    if (!sms) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) { sms = 0; return (int)e; }
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, fn);
        if (e != cudaSuccess) { sms = 0; return (int)e; }
        max_smem -= (int)fa.sharedSizeBytes + 1024;
        if (sms > WR_EP_MAX_GRID) sms = WR_EP_MAX_GRID;
    }
    out->grid = sms;
    out->chunk = (n4 + sms - 1) / sms;
    out->smem = (size_t)out->chunk * 48;
    out->fn = fn;
    if ((int64_t)out->smem > (int64_t)max_smem) return -1000;      // not eligible: the state does not fit
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        if (e != cudaSuccess) return (int)e;
        attr_set = 1;
    }
    return 0;
}

// The owner-computes kernel: slices are whole rows; shared memory holds P / M / V / G of the slice (64 B per float4), the
// int32 ids of `depth` staged steps and the CTA's work list (3 bcap entries at worst).
template <int LPR, int VPL>
static int epoch_owner_config_for(int64_t n_rows, int D, int64_t max_batch, EpochConfig *out) {
    static int sms = 0, max_smem = 0, attr_set = 0;
    const void *fn = (const void *)bprmf_epoch_owner_kernel<LPR, VPL>;
    if (!sms) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) { sms = 0; return (int)e; }
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, fn);
        if (e != cudaSuccess) { sms = 0; return (int)e; }
        max_smem -= (int)fa.sharedSizeBytes + 1024;
        if (sms > WR_EP_MAX_GRID) sms = WR_EP_MAX_GRID;
    }
    if (max_batch > (1 << 20)) return -1000;
    out->grid = sms;
    out->owner = 1;
    out->rows_per_cta = (int)((n_rows + sms - 1) / sms);
    out->chunk = (int64_t)out->rows_per_cta * (D / 4);
    out->bcap = (int)((max_batch + 31) & ~(int64_t)31);
    out->fn = fn;
    const int64_t state = out->chunk * 64, per_stage = (int64_t)out->bcap * 24;      // int64 ids [3][bcap]; two int32 lists = one more
    int depth = EP_STAGE_DEPTH;
    while (depth >= 2 && state + (depth + 1) * per_stage > (int64_t)max_smem) --depth;
    if (depth < 2) return -1000;
    out->depth = depth;
    out->smem = (size_t)(state + (depth + 1) * per_stage);
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        if (e != cudaSuccess) return (int)e;
        attr_set = 1;
    }
    return 0;
}

static int epoch_owner_config(int64_t n_elems, int D, int64_t max_batch, EpochConfig *cfg) {
    const int64_t n_rows = n_elems / D;
    switch (D) {     // more float4 per lane than the two-barrier kernel: more entries in flight per CTA
        case 16: return epoch_owner_config_for<2, 2>(n_rows, D, max_batch, cfg);
        case 32: return epoch_owner_config_for<4, 2>(n_rows, D, max_batch, cfg);
        case 64: return epoch_owner_config_for<8, 2>(n_rows, D, max_batch, cfg);
        case 128: return epoch_owner_config_for<16, 2>(n_rows, D, max_batch, cfg);
        case 256: return epoch_owner_config_for<32, 2>(n_rows, D, max_batch, cfg);
        default: return -1000;
    }
}

// WR_EPOCH_KERNEL=two_barrier keeps the first resident kernel (profiling / comparison)
static bool epoch_owner_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WR_EPOCH_KERNEL");
        v = (e && strcmp(e, "two_barrier") == 0) ? 0 : 1;
    }
    return v == 1;
}

// 0 = eligible (cfg filled), -1000 = not eligible (use the per-step path), anything else = error
// WR_CTX_KERNEL=owner puts the host-fed context on the one-barrier kernel too (its streaming path is complete and tested,
// tests/test_resident_epoch.py::test_host_fed_owner_every_dim; see epoch_config for why it is not the default there)
static bool ctx_owner_ok() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WR_CTX_KERNEL");
        v = (e && strcmp(e, "owner") == 0) ? 1 : 0;
    }
    return v == 1;
}

// owner_ok: the one-barrier kernel may be chosen.  The host-fed context keeps the two-barrier kernel: with the host waiting
// for every step, what counts is the latency of ONE step from descriptor to completion word, and there the owner form
// loses ~2.7 us (every CTA stages and scans the whole batch before it can start; measured e2e 25.6 -> 28.3 us per step),
// while it wins where steps run back to back (6.4 -> 5.6 us per step).
static int epoch_config(int64_t n_elems, int D, int64_t max_batch, EpochConfig *cfg, bool owner_ok = true) {
    if (n_elems & 3) return -1000;
    memset(cfg, 0, sizeof(*cfg));
    if (owner_ok && epoch_owner_enabled()) {
        const int rco = epoch_owner_config(n_elems, D, max_batch, cfg);
        if (rco != -1000) return rco;
        memset(cfg, 0, sizeof(*cfg));
    }
    int rc;
    switch (D) {
        case 16: rc = epoch_config_for<4, 1>(n_elems >> 2, cfg); break;
        case 32: rc = epoch_config_for<8, 1>(n_elems >> 2, cfg); break;
        case 64: rc = epoch_config_for<16, 1>(n_elems >> 2, cfg); break;
        case 128: rc = epoch_config_for<32, 1>(n_elems >> 2, cfg); break;
        case 256: rc = epoch_config_for<32, 2>(n_elems >> 2, cfg); break;
        default: return -1000;
    }
    if (rc) return rc;
    if (max_batch > (int64_t)cfg->grid * EP_STAGE_CAP) return -1000;
    return 0;
}

static int epoch_launch(const EpochConfig &cfg, EpochParams &p, cudaStream_t st) {
    void *args[] = {&p};
    return (int)cudaLaunchCooperativeKernel(cfg.fn, dim3(cfg.grid), dim3(EP_BLOCK), args, cfg.smem, st);
}

static uint64_t *g_epoch_trace = nullptr, *g_epoch_cta_trace = nullptr;      // wr_debug_epoch_trace

static void epoch_fill(EpochParams &p, const EpochConfig &cfg, float *P, float *M, float *V, float *G, int64_t n_elems,
                       int64_t n_users, int64_t n_items, float gamma, float l2, double beta1, double beta2, float eps,
                       void *ws) {
    memset(&p, 0, sizeof(p));
    p.P = (float4 *)P; p.M = (float4 *)M; p.V = (float4 *)V; p.G = (float4 *)G;
    p.n4 = n_elems >> 2;
    p.chunk = cfg.chunk;
    p.rows_per_cta = cfg.rows_per_cta;
    p.bcap = cfg.bcap;
    p.depth = cfg.depth;
    p.n_users = n_users; p.n_items = n_items;
    p.gamma = gamma; p.l2 = l2;
    p.w1 = (float)(1.0 - beta1); p.beta2 = (float)beta2; p.w2 = (float)(1.0 - beta2); p.eps = eps;
    p.ws = (WrWorkspace *)ws;
    p.trace = g_epoch_trace;
    p.cta_trace = g_epoch_cta_trace;
}

// The host-fed context launches the resident kernel for the largest batch seen so far, at least 2,048 rows, in steps of
// 1,024 (so a stream of ragged batches does not relaunch it); `cur` is the capacity it runs with now (0: none yet).
static inline int64_t ctx_batch_cap(int64_t cur, int64_t B) {
    if (B <= cur) return cur;
    return B < 2048 ? 2048 : (B + 1023) & ~(int64_t)1023;
}

// torch/optim/adam.py evaluates these in Python floats (C doubles, libm pow): the same calls here
static inline void adam_step_scalars(double lr, double beta1, double beta2, double t, float *step_size, float *bc2_sqrt) {
    *step_size = (float)(lr / (1.0 - pow(beta1, t)));
    *bc2_sqrt = (float)pow(1.0 - pow(beta2, t), 0.5);
}

}  // namespace wr

using namespace wr;

extern "C" int wr_debug_epoch_trace(uint64_t *dev_trace, uint64_t *dev_cta_trace) {
    g_epoch_trace = dev_trace;
    g_epoch_cta_trace = dev_cta_trace;
    return WR_OK;
}

extern "C" int wr_bprmf_epoch_form(int64_t n_users, int64_t n_items, int D, int64_t batch_cap, int host_fed) {
    if (n_users <= 0 || n_items <= 0 || batch_cap <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    EpochConfig cfg;
    const int64_t bcap = host_fed ? ctx_batch_cap(0, batch_cap) : batch_cap;
    const int rc = epoch_config((n_users + n_items) * D, D, bcap, &cfg, host_fed ? ctx_owner_ok() : true);
    if (rc == -1000) return 0;
    if (rc > 0) return -1000 - rc;      // a CUDA error (no device): kept apart from the forms
    if (rc < 0) return rc;
    return cfg.owner ? 2 : 1;
}

extern "C" size_t wr_bprmf_epoch_scratch_bytes(int64_t N, int64_t batch) {
    if (N <= 0 || batch <= 0) return 0;
    return (size_t)((N + batch - 1) / batch) * sizeof(StepDesc);
}

int wr_bprmf_step_impl(float *P, float *M, float *V, float *G, const int64_t *user, const int64_t *pos, const int64_t *neg,
                       int64_t B, int D, int64_t n_users, int64_t n_items, float gamma, float l2, double beta1, double beta2,
                       float eps, float step_size, float bc2_sqrt, const float *dev_scalars, float *loss_out, void *ws,
                       void *stream);      // train_kernels.cu: the per-step launches

extern "C" int wr_bprmf_epoch(float *P, float *M, float *V, float *G, const int64_t *ids, int64_t N, int64_t batch,
                              int D, int64_t n_users, int64_t n_items, float gamma, double lr, float l2, double beta1,
                              double beta2, float eps, int64_t adam_t0, float *losses, void *scratch,
                              size_t scratch_bytes, void *ws, void *stream) {
    if (!P || !M || !V || !G || !ids || !losses || !ws) return WR_E_NULL;
    if (N <= 0 || batch <= 0 || adam_t0 < 0 || n_users <= 0 || n_items <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(P) || !wr_aligned16(M) || !wr_aligned16(V) || !wr_aligned16(G)) return WR_E_ALIGN;
    const int64_t steps = (N + batch - 1) / batch;
    cudaStream_t st = (cudaStream_t)stream;
    EpochConfig cfg;
    const int64_t n_elems = (n_users + n_items) * D;
    int rc = steps < (int64_t)EP_COUNT_MASK && scratch && scratch_bytes >= (size_t)steps * sizeof(StepDesc) &&
                     wr_aligned16(scratch)
                 ? epoch_config(n_elems, D, batch, &cfg)
                 : -1000;
    if (rc == 0) {
        // one resident launch: the step descriptors (batch slice, Adam scalars of that step) go up in one copy
        std::vector<StepDesc> desc((size_t)steps);
        for (int64_t s = 0; s < steps; ++s) {
            const int64_t lo = s * batch;
            StepDesc &d = desc[(size_t)s];
            d.ids = ids + lo;
            d.stride = N;
            d.B = (int32_t)(N - lo < batch ? N - lo : batch);
            adam_step_scalars(lr, beta1, beta2, (double)(adam_t0 + s + 1), &d.step_size, &d.bc2_sqrt);
            d.seq = (uint32_t)(s + 1);
        }
        cudaError_t e = cudaMemcpyAsync(scratch, desc.data(), (size_t)steps * sizeof(StepDesc), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return (int)e;       // pageable source: staged before the call returns
        EpochParams p;
        epoch_fill(p, cfg, P, M, V, G, n_elems, n_users, n_items, gamma, l2, beta1, beta2, eps, ws);
        p.desc = (const StepDesc *)scratch;
        p.desc_ring = (uint32_t)steps;
        p.first_step = 0;
        p.preset_count = (uint32_t)steps;
        p.losses = losses;
        return epoch_launch(cfg, p, st);
    }
    if (rc != -1000) return rc;
    int64_t s = 0;
    for (int64_t lo = 0; lo < N; lo += batch, ++s) {
        const int64_t B = N - lo < batch ? N - lo : batch;
        float step_size, bc2_sqrt;
        adam_step_scalars(lr, beta1, beta2, (double)(adam_t0 + s + 1), &step_size, &bc2_sqrt);
        rc = wr_bprmf_step_impl(P, M, V, G, ids + lo, ids + N + lo, ids + 2 * N + lo, B, D, n_users, n_items, gamma, l2,
                                beta1, beta2, eps, step_size, bc2_sqrt, nullptr, losses + s, ws, stream);
        if (rc) return rc;
    }
    return WR_OK;
}

// ---- host-fed training: wr_bprmf_ctx_* --------------------------------------------------------------------------------
constexpr uint32_t CTX_RING = 16;

struct HostRing {                      // one mapped pinned allocation
    StepDesc desc[CTX_RING];
    uint32_t lossq[2 * CTX_RING];      // {step + 1, loss bits} written by the kernel as one 8-byte store
    uint32_t done[CTX_RING];
    uint32_t exit_word;
    uint32_t pad[15];
};

// A step of the context that ran as per-step launches (large tables / batches) signals like a resident step: after the
// step on the same stream, one thread stores its loss word pair, then its completion word, into the mapped ring.
__global__ void ctx_signal_kernel(const float *loss, uint32_t *lossq, uint32_t *done, uint32_t seq) {
    asm volatile("st.relaxed.sys.global.v2.b32 [%0], {%1, %2};" ::"l"(lossq), "r"(seq), "r"(__float_as_uint(*loss)) : "memory");
    __threadfence_system();
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(done), "r"(seq) : "memory");
}

struct wr_bprmf_ctx {
    float *P, *M, *V, *G;
    int64_t n_users, n_items;
    int D;
    float gamma, l2, eps;
    double beta1, beta2, lr;
    void *ws;
    cudaStream_t stream;               // the caller's stream (orders the resident kernel against the caller's other work)
    cudaStream_t kstream;              // the resident kernel's own stream
    cudaEvent_t ev;
    HostRing *hr;                      // mapped pinned
    StepDesc *dev_desc;                // device ring [CTX_RING]
    int64_t *stage_ids;                // mapped pinned [CTX_RING][3 * stage_cap], for id buffers that are not mapped
    int64_t stage_cap;
    int64_t *dev_ids;                  // device [CTX_RING][3 * dev_cap]: where the helper warps put the ids they pull over PCIe
    int64_t dev_cap;
    int64_t bcap;                      // batch capacity the resident kernel is configured for
    float *dev_loss;                   // per-step launches: the step's loss before ctx_signal_kernel forwards it
    uint32_t pushed;                   // steps handed over so far (on either route)
    uint32_t first_live;               // first step the resident kernel (or the next launch) is responsible for; steps
                                       // below it are complete or queued on `stream` as per-step launches
    bool resident;
    uint64_t idle_ns;
    const void *checked[4];
    uint32_t n_checked;
    const void *unmapped[64];
};

extern "C" int wr_bprmf_ctx_create(float *P, float *M, float *V, float *G, int64_t n_users, int64_t n_items, int D,
                                   float gamma, double lr, float l2, double beta1, double beta2, float eps, void *ws,
                                   void *stream, wr_bprmf_ctx **out) {
    if (!P || !M || !V || !G || !ws || !out) return WR_E_NULL;
    if (n_users <= 0 || n_items <= 0) return WR_E_SIZE;
    if (D <= 0 || (D & 3)) return WR_E_DIM;
    if (!wr_aligned16(P) || !wr_aligned16(M) || !wr_aligned16(V) || !wr_aligned16(G)) return WR_E_ALIGN;
    wr_bprmf_ctx *c = new (std::nothrow) wr_bprmf_ctx();
    if (!c) return (int)cudaErrorMemoryAllocation;
    c->P = P; c->M = M; c->V = V; c->G = G;
    c->n_users = n_users; c->n_items = n_items; c->D = D;
    c->gamma = gamma; c->l2 = l2; c->eps = eps; c->beta1 = beta1; c->beta2 = beta2; c->lr = lr;
    c->ws = ws; c->stream = (cudaStream_t)stream;
    c->idle_ns = 5000000ull;           // 5 ms without a new batch: the resident kernel writes its state back and leaves
    void *h = nullptr;
    cudaError_t e = cudaHostAlloc(&h, sizeof(HostRing), cudaHostAllocMapped | cudaHostAllocPortable);
    if (e == cudaSuccess) {
        memset(h, 0, sizeof(HostRing));
        c->hr = (HostRing *)h;
        e = cudaMalloc((void **)&c->dev_desc, CTX_RING * sizeof(StepDesc));
    }
    if (e == cudaSuccess) e = cudaMalloc((void **)&c->dev_loss, sizeof(float));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->kstream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        if (c->hr) cudaFreeHost(c->hr);
        if (c->dev_desc) cudaFree(c->dev_desc);
        if (c->dev_loss) cudaFree(c->dev_loss);
        if (c->kstream) cudaStreamDestroy(c->kstream);
        delete c;
        return (int)e;
    }
    *out = c;
    return WR_OK;
}

// Is p mapped pinned memory?  The driver query costs ~1 us, so answers are remembered per address: 4 positive entries, and
// a direct-mapped table of negatives (a stale negative only costs a copy into the context's own pinned ring).
static int ctx_ids_are_mapped(wr_bprmf_ctx *c, const void *p) {
    for (int i = 0; i < 4; ++i)
        if (c->checked[i] == p) return 1;
    const size_t h = ((uintptr_t)p >> 6) & 63u;
    if (c->unmapped[h] == p) return 0;
    cudaPointerAttributes a;
    bool mapped = false;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
        cudaGetLastError();
    else
        mapped = a.type == cudaMemoryTypeHost && a.devicePointer == p;   // pinned, and the same address on the device
    if (mapped)
        c->checked[c->n_checked++ & 3] = p;
    else
        c->unmapped[h] = p;
    return mapped ? 1 : 0;
}

// The resident kernel has left (closed by us, or idle): its stream is drained and the caller's stream ordered behind it.
static int ctx_retire(wr_bprmf_ctx *c) {
    cudaError_t e = cudaStreamSynchronize(c->kstream);
    c->resident = false;
    if (e != cudaSuccess) return (int)e;
    e = cudaEventRecord(c->ev, c->kstream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c->stream, c->ev, 0);
    return (int)e;
}

static int ctx_launch(wr_bprmf_ctx *c, const EpochConfig &cfg) {
    // order the resident kernel behind whatever the caller's stream has done to the tables so far
    cudaError_t e = cudaEventRecord(c->ev, c->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c->kstream, c->ev, 0);
    // the device descriptor ring still holds the previous launch's descriptors (its close marker among them)
    if (e == cudaSuccess) e = cudaMemsetAsync(c->dev_desc, 0, CTX_RING * sizeof(StepDesc), c->kstream);
    if (e != cudaSuccess) return (int)e;
    EpochParams p;
    epoch_fill(p, cfg, c->P, c->M, c->V, c->G, (c->n_users + c->n_items) * c->D, c->n_users, c->n_items, c->gamma, c->l2,
               c->beta1, c->beta2, c->eps, c->ws);
    p.desc = c->dev_desc;
    p.desc_ring = CTX_RING;
    p.first_step = c->first_live;
    p.host_desc = c->hr->desc;
    p.host_ring = CTX_RING;
    p.host_lossq = c->hr->lossq;
    p.host_done = c->hr->done;
    p.host_exit = &c->hr->exit_word;
    p.idle_ns = c->idle_ns;
    p.dev_ids = c->dev_ids;
    p.dev_ids_cap = c->dev_cap;
    __atomic_store_n(&c->hr->exit_word, 0u, __ATOMIC_RELEASE);
    const int rc = epoch_launch(cfg, p, c->kstream);
    if (rc == 0) c->resident = true;
    return rc;
}

// If the kernel left on its own (idle), take note: steps >= exit_word - 1 belong to the next launch.
static int ctx_check_exit(wr_bprmf_ctx *c) {
    if (!c->resident) return 0;
    const uint32_t x = __atomic_load_n(&c->hr->exit_word, __ATOMIC_ACQUIRE);
    if (!x) return 0;
    c->first_live = x - 1u;
    return ctx_retire(c);
}

static int ctx_wait_word(wr_bprmf_ctx *c, const EpochConfig &cfg, volatile uint32_t *word, uint32_t step) {
    for (uint32_t spins = 0; __atomic_load_n(word, __ATOMIC_ACQUIRE) != step + 1u; ++spins) {
        if ((spins & 0x3ffu) == 0x3ffu) {
            int rc = ctx_check_exit(c);
            if (rc) return rc;
            if (!c->resident) {
                if (__atomic_load_n(word, __ATOMIC_ACQUIRE) == step + 1u) break;
                if (step < c->first_live) {
                    // not the resident kernel's: a per-step launch, whose words the caller's stream writes
                    const cudaError_t e = cudaStreamSynchronize(c->stream);
                    if (e != cudaSuccess) return (int)e;
                    if (__atomic_load_n(word, __ATOMIC_ACQUIRE) == step + 1u) break;
                    return (int)cudaErrorUnknown;                              // finished, yet never signalled
                }
                rc = ctx_launch(c, cfg);
                if (rc) return rc;
            } else if ((spins & 0xfffffu) == 0xfffffu) {
                const cudaError_t q = cudaStreamQuery(c->kstream);
                if (q != cudaSuccess && q != cudaErrorNotReady) return (int)q;
                if (q == cudaSuccess && !__atomic_load_n(&c->hr->exit_word, __ATOMIC_ACQUIRE) &&
                    __atomic_load_n(word, __ATOMIC_ACQUIRE) != step + 1u)
                    return (int)cudaErrorUnknown;                            // the kernel is gone without a word
            }
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    return 0;
}

extern "C" int wr_bprmf_ctx_sync(wr_bprmf_ctx *c) {
    if (!c) return WR_E_NULL;
    if (!c->resident) return WR_OK;
    int rc = ctx_check_exit(c);
    if (rc || !c->resident) return rc;
    // close: a descriptor with B = -1 in the slot of the next step
    const uint32_t s = c->pushed;
    EpochConfig cfg;
    rc = epoch_config((c->n_users + c->n_items) * c->D, c->D, c->bcap > 0 ? c->bcap : 1, &cfg, ctx_owner_ok());
    if (rc) return rc;
    if (s >= CTX_RING) {
        rc = ctx_wait_word(c, cfg, &c->hr->done[s % CTX_RING], s - CTX_RING);
        if (rc) return rc;
        if (!c->resident) return WR_OK;       // it idled out meanwhile (and was not needed again)
    }
    StepDesc *d = &c->hr->desc[s % CTX_RING];
    d->ids = nullptr; d->stride = 0; d->B = -1; d->step_size = 0.f; d->bc2_sqrt = 0.f;
    __atomic_store_n(&d->seq, s + 1u, __ATOMIC_RELEASE);
    rc = ctx_retire(c);
    c->first_live = c->pushed;
    __atomic_store_n(&d->seq, 0u, __ATOMIC_RELEASE);      // the slot will carry a real step s later
    return rc;
}

extern "C" int wr_bprmf_ctx_destroy(wr_bprmf_ctx *c) {
    if (!c) return WR_E_NULL;
    wr_bprmf_ctx_sync(c);
    cudaStreamSynchronize(c->stream);
    cudaStreamDestroy(c->kstream);
    cudaEventDestroy(c->ev);
    cudaFreeHost(c->hr);
    if (c->stage_ids) cudaFreeHost(c->stage_ids);
    if (c->dev_ids) cudaFree(c->dev_ids);
    cudaFree(c->dev_desc);
    cudaFree(c->dev_loss);
    delete c;
    return WR_OK;
}

extern "C" int wr_bprmf_ctx_wait(wr_bprmf_ctx *c, int64_t step, int wait, float *host_loss_out) {
    if (!c) return WR_E_NULL;
    if (step < 0 || step >= (int64_t)c->pushed || (int64_t)c->pushed - step > (int64_t)CTX_RING || wait < 1 || wait > 2)
        return WR_E_SIZE;
    EpochConfig cfg;
    int rc = epoch_config((c->n_users + c->n_items) * c->D, c->D, c->bcap > 0 ? c->bcap : 1, &cfg, ctx_owner_ok());
    // -1000: the context never ran resident, so every step is below first_live and cfg is never launched
    if (rc && rc != -1000) return rc;
    const uint32_t s = (uint32_t)step;
    rc = ctx_wait_word(c, cfg, wait == 2 ? &c->hr->lossq[2 * (s % CTX_RING)] : &c->hr->done[s % CTX_RING], s);
    if (rc) return rc;
    if (host_loss_out) memcpy(host_loss_out, (const void *)&c->hr->lossq[2 * (s % CTX_RING) + 1], sizeof(float));
    return WR_OK;
}

// Pageable (or unmapped) ids go into slot s of the context's own pinned ring -- the host half of the H2D transfer; *ids
// is what the kernels read.  The slot's previous tenant is complete (the caller has waited for it).
static int ctx_stage_ids(wr_bprmf_ctx *c, const int64_t *host_ids, int64_t B, uint32_t s, const int64_t **ids) {
    *ids = host_ids;
    if (wr_aligned16(host_ids) && ctx_ids_are_mapped(c, host_ids)) return WR_OK;
    if (B > c->stage_cap) {
        int rc = wr_bprmf_ctx_sync(c);
        if (rc) return rc;
        const cudaError_t q = cudaStreamSynchronize(c->stream);     // per-step launches may still read the old ring
        if (q != cudaSuccess) return (int)q;
        if (c->stage_ids) cudaFreeHost(c->stage_ids);
        c->stage_ids = nullptr;
        c->stage_cap = ((B < 4096 ? 4096 : B) + 15) & ~(int64_t)15;
        const cudaError_t e = cudaHostAlloc((void **)&c->stage_ids, (size_t)CTX_RING * 3 * c->stage_cap * sizeof(int64_t),
                                            cudaHostAllocMapped | cudaHostAllocPortable);
        if (e != cudaSuccess) { c->stage_cap = 0; return (int)e; }
    }
    int64_t *slot = c->stage_ids + (size_t)(s % CTX_RING) * 3 * c->stage_cap;
    memcpy(slot, host_ids, (size_t)(3 * B) * sizeof(int64_t));
    *ids = slot;
    return WR_OK;
}

extern "C" int wr_bprmf_ctx_step(wr_bprmf_ctx *c, const int64_t *host_ids, int64_t B, int64_t adam_t, int wait,
                                 float *host_loss_out) {
    if (!c || !host_ids) return WR_E_NULL;
    if (B <= 0 || adam_t <= 0 || B > INT32_MAX) return WR_E_SIZE;
    float step_size, bc2_sqrt;
    adam_step_scalars(c->lr, c->beta1, c->beta2, (double)adam_t, &step_size, &bc2_sqrt);
    const int64_t n_elems = (c->n_users + c->n_items) * c->D;
    const int D = c->D;
    EpochConfig cfg;
    // the resident kernel stages whole batches in shared memory: it is launched for the largest batch seen so far and
    // relaunched when a larger one arrives
    const int64_t bcap = ctx_batch_cap(c->bcap, B);
    int rc = epoch_config(n_elems, D, bcap, &cfg, ctx_owner_ok());
    if (rc == 0 && bcap != c->bcap) {
        rc = wr_bprmf_ctx_sync(c);        // (still configured for the old size: closes the running kernel, if any)
        if (rc) return rc;
        c->bcap = bcap;
    }
    if (rc != 0 && rc != -1000) return rc;
    const bool per_step = rc == -1000;
    if (per_step) {
        // large tables / batches: per-step launches on the caller's stream.  The step still takes the next step number
        // and ring slot, so wr_bprmf_ctx_wait finds it like any other step.
        rc = wr_bprmf_ctx_sync(c);
        if (rc) return rc;
    } else {
        rc = ctx_check_exit(c);
        if (rc) return rc;
    }
    const uint32_t s = c->pushed;
    if (s >= EP_COUNT_MASK - 1u) return WR_E_SIZE;
    if (s >= CTX_RING) {                 // the slot's previous tenant (step s - CTX_RING) must be complete
        rc = ctx_wait_word(c, cfg, &c->hr->done[s % CTX_RING], s - CTX_RING);
        if (rc) return rc;
    }
    if (!per_step && B > c->dev_cap) {   // (re)size the device-side id ring; the kernel must not be running on the old one
        rc = wr_bprmf_ctx_sync(c);
        if (rc) return rc;
        if (c->dev_ids) cudaFree(c->dev_ids);
        c->dev_ids = nullptr;
        c->dev_cap = ((B < 4096 ? 4096 : B) + 15) & ~(int64_t)15;
        const cudaError_t e = cudaMalloc((void **)&c->dev_ids, (size_t)CTX_RING * 3 * c->dev_cap * sizeof(int64_t));
        if (e != cudaSuccess) { c->dev_cap = 0; return (int)e; }
    }
    const int64_t *ids = host_ids;
    rc = ctx_stage_ids(c, host_ids, B, s, &ids);
    if (rc) return rc;
    if (per_step) {
        // the kernels read the ids straight from mapped pinned memory; the loss and completion words reach the same
        // slots the resident kernel writes
        rc = wr_bprmf_step_impl(c->P, c->M, c->V, c->G, ids, ids + B, ids + 2 * B, B, D, c->n_users, c->n_items,
                                c->gamma, c->l2, c->beta1, c->beta2, c->eps, step_size, bc2_sqrt, nullptr, c->dev_loss,
                                c->ws, c->stream);
        if (rc) return rc;
        ctx_signal_kernel<<<1, 1, 0, c->stream>>>(c->dev_loss, &c->hr->lossq[2 * (s % CTX_RING)],
                                                   &c->hr->done[s % CTX_RING], s + 1u);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
        c->pushed = s + 1u;
        c->first_live = s + 1u;
        if (!wait) return WR_OK;
        e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) return (int)e;
        if (__atomic_load_n(&c->hr->done[s % CTX_RING], __ATOMIC_ACQUIRE) != s + 1u) return (int)cudaErrorUnknown;
        if (host_loss_out) memcpy(host_loss_out, (const void *)&c->hr->lossq[2 * (s % CTX_RING) + 1], sizeof(float));
        return WR_OK;
    }
    StepDesc *d = &c->hr->desc[s % CTX_RING];
    d->ids = ids; d->stride = B; d->B = (int32_t)B; d->step_size = step_size; d->bc2_sqrt = bc2_sqrt;
    __atomic_store_n(&d->seq, s + 1u, __ATOMIC_RELEASE);
    c->pushed = s + 1u;
    if (!c->resident) {
        rc = ctx_launch(c, cfg);
        if (rc) return rc;
    }
    if (!wait) return WR_OK;
    rc = ctx_wait_word(c, cfg, wait == 2 ? &c->hr->lossq[2 * (s % CTX_RING)] : &c->hr->done[s % CTX_RING], s);
    if (rc) return rc;
    if (host_loss_out) memcpy(host_loss_out, (const void *)&c->hr->lossq[2 * (s % CTX_RING) + 1], sizeof(float));
    return WR_OK;
}
