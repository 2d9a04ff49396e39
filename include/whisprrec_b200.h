/* whisprrec_b200.h -- C-ABI of libwhisprrec_b200.so (sm_100a).
 *
 * The reference (HeyWeCome/WhisprRec) has no FFI: its hot path is a chain of PyTorch calls made from
 * Python classes.  Each entry point below replaces the chain of torch ops at the cited reference lines
 * (paths relative to the reference checkout, src/...).  INTEGRATION.md shows the ctypes stub a reference
 * maintainer would add at each site.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name starts with `host_`;
 *   - tables are row-major fp32 [rows, D]; ids are int64 (what `collate_batch` hands to the model,
 *     models/BaseModel.py:96-127); CSR column / history indices are int32, row pointers int64;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it and never syncs the
 *     host (wr_status is the one exception and says so);
 *   - `ws` is a caller-owned device scratch block of wr_workspace_bytes() bytes, zeroed once with
 *     wr_workspace_init; one workspace per stream;
 *   - return value: 0 ok, <0 argument error (WR_E_*), >0 a cudaError_t from the launch;
 *   - D must be a multiple of 4 (128-bit row accesses); other sizes return WR_E_DIM.
 *   - there is no CPU path: on a machine without an sm_100 device every compute call returns the CUDA error.
 */
#ifndef WHISPRREC_B200_H
#define WHISPRREC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WR_VERSION 100

#define WR_OK 0
#define WR_E_NULL (-1)   /* a required pointer is NULL */
#define WR_E_SIZE (-2)   /* a negative / inconsistent size */
#define WR_E_DIM (-3)    /* embedding size not supported (D % 4 != 0 or D > 512) */
#define WR_E_TOPK (-4)   /* k outside [1, 32] ([1, 256] for the _long calls, at precision 0 or 2 only) */
#define WR_E_ALIGN (-5)  /* a table pointer is not 16-byte aligned */
#define WR_E_PRECISION (-6) /* unknown / unavailable scoring precision */

/* bits of the device-side status word (wr_status) */
#define WR_STATUS_INDEX_OUT_OF_RANGE 1u /* an id outside its table: the row was skipped (torch raises IndexError) */
#define WR_STATUS_PEER_TIMEOUT 2u       /* a cross-GPU wait gave up after WR_PEER_TIMEOUT_NS: a peer never arrived
                                           (crashed or out of step); results of that step are invalid */
#define WR_STATUS_EVAL_OVERFLOW 4u      /* precision-2 evaluation: more score/target near-ties than the candidate list
                                           holds (degenerate tables, e.g. all rows equal); ranks are incomplete -- rerun
                                           with precision 0 */
#define WR_STATUS_TOPK_OVERFLOW 8u      /* precision-2 top-k: a row had more list candidates than its segment holds; its
                                           list is returned as topk_idx[r, 0] = -2 -- rerun those rows with precision 0.
                                           Long lists (wr_eval_rank_topk_long): such rows were finished on the device;
                                           their lists are exact */
#define WR_PEER_TIMEOUT_NS 20000000000ull

int wr_version(void);
const char *wr_error_string(int code);

size_t wr_workspace_bytes(void);
int wr_workspace_init(void *ws, void *stream);
/* Copies the status word to *host_status and clears it.  SYNCHRONISES the stream. */
int wr_status(void *ws, uint32_t *host_status, void *stream);

/* ---- training ---------------------------------------------------------------------------------------
 * wr_bpr_fwd_bwd: models/general/BPRMF.py:69-80 (gather, row dots), utils/loss.py:33-39 (BPRLoss) and the
 * autograd backward BaseRunner.py:198 triggers, in one launch.
 *   loss = -mean_b log(gamma + sigmoid(<U[u_b],I[p_b]> - <U[u_b],I[n_b]>))
 *   c_b  = grad_scale * dloss/ds+_b ;  gU[u_b] += c_b (I[p_b]-I[n_b]);  gI[p_b] += c_b U[u_b];  gI[n_b] -= c_b U[u_b]
 * gU/gI are ACCUMULATED into (they must hold zeros or an earlier partial gradient; wr_adam_l2_sweep leaves
 * them zeroed).  U/I may be the ego tables (BPRMF) or the pooled tables (LightGCN.py:155-162, grad_scale =
 * 1/(L+1) folds the mean-pool adjoint in).  loss_out[0] is overwritten (accumulate_loss = 0) or added to.
 */
int wr_bpr_fwd_bwd(const float *U, const float *I, const int64_t *user, const int64_t *pos, const int64_t *neg,
                   int64_t B, int D, int64_t n_users, int64_t n_items, float gamma, float grad_scale,
                   float *gU, float *gI, float *loss_out, int accumulate_loss, void *ws, void *stream);

/* wr_embloss_fwd_bwd: utils/loss.py:83-98 (EmbLoss, require_pow=False) as called at LightGCN.py:165-175.
 *   reg = (||U0[user]||_F + ||I0[pos]||_F + ||I0[neg]||_F) / B ;  loss_out[0] += reg_weight * reg
 *   gU0[u_b] += reg_weight/B * U0[u_b]/||U0[user]||_F   (and likewise for pos / neg rows)
 * Two launches: the norms are batch-global and must exist before the gradient.
 */
int wr_embloss_fwd_bwd(const float *U0, const float *I0, const int64_t *user, const int64_t *pos,
                       const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items, float reg_weight,
                       float *gU0, float *gI0, float *loss_out, void *ws, void *stream);

/* wr_adam_l2_sweep: torch.optim.Adam(weight_decay=l2).step() as built at helpers/BaseRunner.py:120-124 and
 * called at :199 (torch/optim/adam.py _single_tensor_adam), plus the zero_grad of :196, fused in one sweep
 * over ALL rows (dense Adam: every row moves every step).
 *   g += l2 p;  m += (1-b1)(g-m);  v = b2 v + (1-b2) g g;  p -= step_size * m / (sqrt(v)/bc2_sqrt + eps);  g = 0
 * step_size = lr/(1-b1^t) and bc2_sqrt = sqrt(1-b2^t) are evaluated in double by the caller as torch does;
 * the betas are doubles because torch forms 1-beta in double before rounding it for the fp32 kernels.
 * If dev_scalars != NULL, {step_size, bc2_sqrt} are read from that device array instead (lets a captured
 * CUDA graph be replayed for later steps).
 */
int wr_adam_l2_sweep(float *P, float *M, float *V, float *G, int64_t n_elems, float l2, double beta1, double beta2,
                     float eps, float step_size, float bc2_sqrt, const float *dev_scalars, void *stream);

/* wr_bprmf_step: one whole iteration of BaseRunner.fit for BPRMF (BaseRunner.py:196-199: zero_grad, predict,
 * backward, Adam.step) on the fused table P = [U; I] ([n_users + n_items, D], M / V / G alike).  Tables of up to
 * 8 Mi elements take ONE cooperative launch (L2 prefetch of the CTA's P / M / V / G spans, BPR forward+backward, grid
 * barrier, Adam+L2 with the gradient re-zeroed); larger ones are wr_bpr_fwd_bwd followed by wr_adam_l2_sweep.  Same
 * arithmetic either way.  loss_out[0] is overwritten.  (A whole epoch of such steps: wr_bprmf_epoch.)
 */
int wr_bprmf_step(float *P, float *M, float *V, float *G, const int64_t *user, const int64_t *pos,
                  const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items, float gamma, float l2,
                  double beta1, double beta2, float eps, float step_size, float bc2_sqrt, const float *dev_scalars,
                  float *loss_out, void *ws, void *stream);

/* Row-marked variants for tables too large for the caches, where the sweep is HBM-bound.  BPRMF's gradient is zero
 * outside the 3 B rows of the batch (models/general/BPRMF.py:41-53: only the gathered rows enter the loss), so `touched`
 * -- ceil(n_rows / 32) uint32 words of DEVICE memory, bit r = row r of G is non-zero, ALL ZERO between steps -- lets
 * the sweep skip the read and the re-zeroing of every other gradient row: 24 bytes of traffic per parameter instead
 * of 32, results identical bit for bit.
 *   wr_mark_rows             sets the bits of a batch (rows user[b], n_users + pos[b], n_users + neg[b])
 *   wr_adam_l2_sweep_marked  wr_adam_l2_sweep over n_rows x D that reads G only where a bit is set; clears the map
 *   wr_inbox_scatter_marked  wr_inbox_scatter that also sets the bit of every owner-local row it adds into
 *   wr_bprmf_step_marked     wr_bprmf_step on the three above (cache-sized tables: the single launch, map untouched)
 */
int wr_mark_rows(const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B, int64_t n_users,
                 int64_t n_items, uint32_t *touched, void *stream);
int wr_adam_l2_sweep_marked(float *P, float *M, float *V, float *G, int64_t n_rows, int D, uint32_t *touched, float l2,
                            double beta1, double beta2, float eps, float step_size, float bc2_sqrt,
                            const float *dev_scalars, void *stream);
int wr_inbox_scatter_marked(float *G, const float *inbox_rows, int32_t *inbox_idx, int world, int64_t cap, int D,
                            uint32_t *touched, void *stream);
int wr_bprmf_step_marked(float *P, float *M, float *V, float *G, uint32_t *touched, const int64_t *user,
                         const int64_t *pos, const int64_t *neg, int64_t B, int D, int64_t n_users, int64_t n_items,
                         float gamma, float l2, double beta1, double beta2, float eps, float step_size, float bc2_sqrt,
                         const float *dev_scalars, float *loss_out, void *ws, void *stream);

/* wr_bprmf_epoch: the step loop of BaseRunner.fit (BaseRunner.py:194-200) in one call: batch s is columns
 * [s * batch, min(N, (s + 1) * batch)) of ids[3][N] (DEVICE, rows user / pos / neg), Adam's t runs from adam_t0 + 1,
 * losses[s] (DEVICE, ceil(N / batch) floats) receives the loss of step s.  When the Adam state fits in the SMs' shared
 * memory (48 B per 4 parameters, ~29 MB over 148 SMs), D is 16 / 32 / 64 / 128 / 256 and batch <= 128 x SMs, the
 * whole epoch is ONE launch of the resident kernel (csrc/epoch_kernel.cu): the Adam moments stay in shared memory from the first step
 * to the last, the next steps' ids are staged by a helper warp per CTA while the current step runs, two grid barriers
 * per step; otherwise one wr_bprmf_step per batch.  scratch: 16-byte aligned DEVICE memory of
 * wr_bprmf_epoch_scratch_bytes(N, batch) bytes (the per-step descriptors: batch slice + Adam scalars of that step,
 * evaluated in double on the host as torch does); NULL forces the per-step form.  Launches only; nothing is synchronised.
 */
size_t wr_bprmf_epoch_scratch_bytes(int64_t N, int64_t batch);
/* Which form trains BPRMF on a table of n_users + n_items rows of size D with batches of at most batch_cap rows:
 * 2 = the owner-computes resident kernel (one grid barrier per step), 1 = the two-barrier resident kernel, 0 = one
 * wr_bprmf_step launch per batch; a negative error otherwise (WR_E_SIZE / WR_E_DIM for bad arguments, -1000 - the CUDA
 * error when the device cannot be queried).  host_fed = 0 answers for wr_bprmf_epoch (with its scratch given),
 * host_fed != 0 for a step of batch_cap rows on a fresh wr_bprmf_ctx (which sizes the kernel for >= 2,048 rows, in
 * steps of 1,024).  The same decision the calls make, WR_EPOCH_KERNEL and WR_CTX_KERNEL included. */
int wr_bprmf_epoch_form(int64_t n_users, int64_t n_items, int D, int64_t batch_cap, int host_fed);
/* Profiling aid: with a DEVICE buffer of 8 x uint64 per step set here (NULL switches it off), every later launch of the
 * resident kernel records %globaltimer stamps per step: [0] step start, [1] BPR phase done, [2] past grid barrier 1,
 * [3] Adam phase done, [4] past grid barrier 2 (CTA 0), [5] descriptor seen by the poller, [6] ids staged (CTA 0),
 * [7] completion word written (streaming).  scripts/prof_resident.py prints the breakdown. */
int wr_debug_epoch_trace(uint64_t *dev_trace, uint64_t *dev_cta_trace /* nullable: [step][CTA][4], both barriers of every CTA */);
/* Profiling aid: with a DEVICE buffer of 8 x uint64 per CTA set here (NULL switches it off), every later one-GPU launch
 * of the single-launch step (wr_bprmf_step on cache-sized tables, D <= 128) records %globaltimer stamps of thread 0 of every CTA:
 * [0] entry, [1] ids landed, [2] rows landed, [3] REDs issued, [4] arrived at the grid barrier, [5] barrier passed,
 * [6] Adam operands landed, [7] exit.  The buffer needs 8 x (CTAs of the launch) words (<= 8 x 2048).
 * scripts/prof_step_phases.py prints the breakdown. */
int wr_debug_step_trace(uint64_t *dev_trace);
int wr_bprmf_epoch(float *P, float *M, float *V, float *G, const int64_t *ids, int64_t N, int64_t batch, int D,
                   int64_t n_users, int64_t n_items, float gamma, double lr, float l2, double beta1, double beta2,
                   float eps, int64_t adam_t0, float *losses, void *scratch, size_t scratch_bytes, void *ws,
                   void *stream);

/* wr_bprmf_step_host: the same iteration fed from the HOST, i.e. utils.batch_to_gpu (utils/utils.py:33-37) +
 * the step + `loss.detach().cpu()` (BaseRunner.py:200).  host_ids: pinned [3, B] int64 (user, pos, neg rows);
 * dev_ids: device staging of the same shape; host_loss: pinned float that receives the batch loss.
 * sync != 0 waits for the stream before returning (the reference syncs on every step).
 */
int wr_bprmf_step_host(const int64_t *host_ids, int64_t *dev_ids, float *host_loss, float *P, float *M, float *V,
                       float *G, int64_t B, int D, int64_t n_users, int64_t n_items, float gamma, float l2,
                       double beta1, double beta2, float eps, float step_size, float bc2_sqrt, float *loss_out,
                       void *ws, void *stream, int sync);

/* wr_bprmf_ctx_*: host-fed training without a launch, a copy-engine hop or a stream synchronisation per step
 * (utils.batch_to_gpu, utils/utils.py:33-37 + BaseRunner.py:196-200 for a loop whose batches are produced on the host).
 * The first wr_bprmf_ctx_step launches the RESIDENT kernel (csrc/epoch_kernel.cu, streaming mode) on the context's own
 * stream; from then on a step is: the host writes a 32-byte descriptor (id buffer, rows, Adam scalars of step adam_t,
 * evaluated in double exactly as torch does) into a ring in mapped pinned memory; a poller warp on the GPU picks it up,
 * helper warps pull the ids out of pinned host memory (that is the H2D transfer), the step runs, and the loss and two
 * sequence words are stored back into mapped host memory (the D2H transfer):
 *   wait = 1  returns when the whole step is complete (every parameter updated);
 *   wait = 2  returns as soon as the batch loss is out (the Adam phase may still be running);
 *   wait = 0  returns at once; up to 16 steps may be in flight, wr_bprmf_ctx_wait(step, ...) collects a loss later
 *             (step = 0 for the context's first wr_bprmf_ctx_step, 1 for the next, ...).
 * host_ids: [3, B] int64.  Mapped pinned memory (torch `.pin_memory()`) is read in place and must stay untouched until
 * the step is complete; anything else is first copied into the context's own pinned ring (the collate copy).
 * The kernel writes M / V back and leaves when wr_bprmf_ctx_sync / wr_bprmf_ctx_destroy close it, or by itself after 5 ms
 * without a new batch (the next step relaunches it).  WHILE IT IS RESIDENT THE ADAM MOMENTS LIVE IN SHARED MEMORY: call
 * wr_bprmf_ctx_sync before anything else reads M / V or writes the tables.  Tables and batches that do not qualify for
 * the resident kernel (wr_bprmf_epoch_form with host_fed = 1 returns 0) run as one launch per step on `stream`; such a
 * step takes the next step number like any other, so wr_bprmf_ctx_wait works after any mix of the two routes.
 */
typedef struct wr_bprmf_ctx wr_bprmf_ctx;
int wr_bprmf_ctx_create(float *P, float *M, float *V, float *G, int64_t n_users, int64_t n_items, int D, float gamma,
                        double lr, float l2, double beta1, double beta2, float eps, void *ws, void *stream,
                        wr_bprmf_ctx **out);
int wr_bprmf_ctx_step(wr_bprmf_ctx *ctx, const int64_t *host_ids, int64_t B, int64_t adam_t, int wait,
                      float *host_loss_out);
int wr_bprmf_ctx_wait(wr_bprmf_ctx *ctx, int64_t step, int wait, float *host_loss_out);
int wr_bprmf_ctx_sync(wr_bprmf_ctx *ctx);
int wr_bprmf_ctx_destroy(wr_bprmf_ctx *ctx);

/* ---- SGL (SURVEY.md section 8 f-3; models/general/SGL.py) -------------------------------------------------------
 * The three propagations of a step are wr_csr_spmm on the main graph and on the two edge-dropout views (which are not
 * symmetric: the backward pass takes the transposed CSR), EmbLoss is wr_embloss_fwd_bwd; what is new:
 * wr_bpr_logsig_sum_fwd_bwd: SGL.py:176-185, loss_out (+)= sum_b -logsigmoid(<U[u_b],I[p_b]> - <U[u_b],I[n_b]>) (a sum,
 *   not a mean); gradients as wr_bpr_fwd_bwd, scaled by grad_scale.
 * wr_infonce_fwd_bwd: SGL.py:196-231 for one block of rows (users of the batch against all users, or positive items
 *   against all items), forward and backward:
 *     a_b = normalize(T1[idx_b]), t_j = normalize(T2[j]) (F.normalize, eps 1e-12), z_b = sum_j exp(a_b . t_j / tau)
 *     loss_out[0] += weight * sum_b (log z_b - a_b . t_{idx_b} / tau)
 *     dT1[idx_b] += grad_scale * dL/dT1[idx_b] (RED per occurrence), dT2[j] += grad_scale * dL/dT2[j] for every j
 *   T1 / T2 / dT1 / dT2: [N, D] fp32 blocks of the pooled view tables and their gradients; D <= 256 (WR_E_DIM above).
 *   The [B, N] contraction is streamed as fp32 FMA tiles in two passes over the table (row sums, then the weights
 *   recomputed for both gradient products); no buffer grows with B x N, so any catalogue size runs.  The loss is the
 *   same bits from call to call; the gradients are summed with REDs.
 *   scratch: wr_infonce_scratch_bytes(B, N, D) bytes of device memory, O((B + N) D) (0 for arguments the call refuses).
 */
int wr_bpr_logsig_sum_fwd_bwd(const float *U, const float *I, const int64_t *user, const int64_t *pos, const int64_t *neg,
                              int64_t B, int D, int64_t n_users, int64_t n_items, float grad_scale, float *gU, float *gI,
                              float *loss_out, int accumulate_loss, void *ws, void *stream);
size_t wr_infonce_scratch_bytes(int64_t B, int64_t N, int D);
int wr_infonce_fwd_bwd(const float *T1, const float *T2, const int64_t *idx, int64_t B, int64_t N, int D, float tau,
                       float weight, float grad_scale, float *dT1, float *dT2, float *loss_out, void *scratch,
                       size_t scratch_bytes, void *ws, void *stream);

/* ---- LightGCN propagation ------------------------------------------------------------------------------
 * wr_csr_norm_weights: the value recipe of LightGCN.py:89-97: val[e] = fl32(fl32(dinv[row] * 1) * dinv[col]).
 * dinv = np.power(fp32(deg) + 1e-10, -0.5) comes from the caller (NumPy's fp32 pow is not correctly rounded,
 * so only the same NumPy call reproduces the reference bit for bit).
 */
int wr_csr_norm_weights(const int64_t *rowptr, const int32_t *col, const float *dinv, int64_t N, float *val,
                        void *stream);

/* wr_csr_spmm: one `torch.sparse.mm(norm_adj, E)` of LightGCN.py:139 fused with the stack/mean of :142-143.
 *   y[r]       = sum_e val[e] * X[col[e]]  (+ add[r] if add != NULL)
 *   Y[r]       = y[r]                                   if Y != NULL
 *   acc_out[r] = (acc_in[r] + y[r]) / acc_div           if acc_out != NULL
 * The backward pass of the propagation is the same call (the adjacency is symmetric): H <- A H + G'.
 * zero_add != 0 clears add[r] after reading it (recycles the pooled-gradient buffer for the next step).
 * X must not alias Y / acc_out.
 */
/* wr_csr_build: the graph construction of LightGCN.py:54-88 on the device (SURVEY.md section 8 f-2).  From E (user, item)
 * pairs (int64, any order, duplicates allowed -- the reference builds R from per-user sets, so a pair counts once) it
 * produces the CSR STRUCTURE of the [N, N] bipartite adjacency [[0, R], [R^T, 0]], N = n_users + n_items:
 *   rowptr [N + 1] int64;  col [2 E] int32 (the first *nnz_out entries are used), ascending inside every row:
 *   user row u lists n_users + i for its items i, item row i lists its users;  *nnz_out (DEVICE) = 2 x distinct pairs.
 * Hand-written and deterministic: stable LSD radix sort of (row << 32 | col) keys (8-bit digits, only the digits that
 * can be non-zero; per-tile histograms, multi-level exclusive scan, match-any ranked scatter), adjacent-unique
 * compaction, row pointers from the key boundaries -- no atomics on the output.  Ids outside their table raise
 * WR_STATUS_INDEX_OUT_OF_RANGE and are dropped.  The fp32 weights are a separate step because d^-1/2 must come from the
 * reference's own NumPy call to match it bit for bit: degrees = diff(rowptr) -> np.power(fp32(deg) + 1e-10, -0.5) ->
 * wr_csr_norm_weights.  scratch: wr_csr_build_scratch_bytes(E) bytes of device memory (two key buffers + histograms).
 */
size_t wr_csr_build_scratch_bytes(int64_t E);
int wr_csr_build(const int64_t *edge_u, const int64_t *edge_i, int64_t E, int64_t n_users, int64_t n_items,
                 int64_t *rowptr, int32_t *col, int64_t *nnz_out, void *scratch, size_t scratch_bytes, void *ws,
                 void *stream);

/* wr_subgraph_csr: SGL's edge-dropout views on the device (utils/augmentor.py:77-111, SGL.py:67-79): the CSR structure
 * (transpose = 0) or the structure of the TRANSPOSE (transpose = 1) of the sub-graph that keeps edges keep[0..K) (edge
 * numbers in CSR order, which is the order of `adj_matrix.nonzero()` in the reference; they come from Python's random
 * stream: wr_pyrandom_sample) of the square CSR matrix (rowptr, col) with n_rows rows.  out_rowptr [n_rows + 1], out_col
 * [K], *nnz_out (DEVICE) = entries kept.  The views are not symmetric (the two directions of an edge are dropped
 * independently), so the backward pass of a propagation needs the transpose.  Same radix-sort machinery and scratch size
 * rule as wr_csr_build; weights: row degrees -> the reference's NumPy d^-1/2 -> wr_csr_norm_weights on either structure.
 */
size_t wr_subgraph_csr_scratch_bytes(int64_t K);
int wr_subgraph_csr(const int64_t *rowptr, const int32_t *col, int64_t n_rows, const int64_t *keep, int64_t K,
                    int transpose, int64_t *out_rowptr, int32_t *out_col, int64_t *nnz_out, void *scratch,
                    size_t scratch_bytes, void *ws, void *stream);

typedef struct wr_spmm_plan {
    /* HOST struct of DEVICE pointers: how rows with more than long_threshold non-zeros are cut into slices so
     * that no warp walks more than one slice (power-law graphs: a 10^6-edge item row would otherwise be the tail
     * of every launch).  Built once per graph by the caller (whisprrec_b200/_lib.py SpmmPlan does it in NumPy). */
    int64_t long_threshold;       /* rows with more non-zeros than this are split */
    int64_t n_chunks, n_long;     /* number of slices, number of split rows */
    const int32_t *chunk_row;     /* [n_chunks] row a slice belongs to */
    const int64_t *chunk_beg;     /* [n_chunks] first edge of the slice */
    const int32_t *chunk_len;     /* [n_chunks] edges in the slice */
    const int32_t *chunk_slot;    /* [n_chunks] index of the split row in the slot arrays */
    const int32_t *slot_chunks;   /* [n_long] slices per split row */
    int32_t *slot_arrivals;       /* [n_long] zeroed; left zeroed by every call */
    float *slot_partial;          /* [n_long, D] zeroed; left zeroed by every call */
    const uint32_t *hot_bits;     /* nullable: bitmap over the N columns; rows of X whose bit is set are loaded with an L2
                                     evict_last policy, the col / val streams with evict_first.  For tables far larger than
                                     L2: mark the highest-degree nodes, as many as fit in ~2/3 of L2 */
    const uint32_t *x_rows;       /* nullable, per call: bitmap over the N columns; a row of X whose bit is CLEAR is taken as
                                     zero and is not fetched (the first backward propagation: the pooled gradient of a
                                     batch is zero outside the batch's 3 B rows, LightGCN.py:150-163).  Same result bit for
                                     bit as reading the zeros.  Takes precedence over hot_bits. */
} wr_spmm_plan;

int wr_csr_spmm(const int64_t *rowptr, const int32_t *col, const float *val, int64_t N, int D, const float *X,
                float *Y, float *add, int zero_add, const float *acc_in, float *acc_out, float acc_div,
                const wr_spmm_plan *host_plan /* nullable */, void *stream);

/* ---- full-ranking evaluation ---------------------------------------------------------------------------
 * wr_eval_rank_topk: BPRMF.py:82-91 / LightGCN.py:177-187 (S = U[user] I^T), BaseRunner.py:238 (target
 * gather), :246-255 (history mask), :72-73 (rank) without materialising S.
 *   target[r] = <U[user_r], I[pos_r]>
 *   rank[r]   = 1 + #{ j not in hist(user_r) : <U[user_r], I[j]> > target[r] }
 *   topk_idx[r,:k], topk_val[r,:k] = the k best unmasked items, best first, ties to the lower id
 *                                    (unfilled slots: idx -1, val -inf); pass NULL to skip.
 * hist_ptr/hist_idx: CSR of the sorted union train_clicked_set U residual_clicked_set per user.
 * scores_out: optional dense fp32 [R, n_items] copy of S, unmasked -- what full_predict returns; NULL on the
 *             fast path (the point of the fusion is not to write it).
 * precision 0: fp32 FMA chains over d = 0..D-1 for every score (target included), so comparisons are
 * consistent; D in {16, 32, 64, 128, 256}.  precision 1: bf16 operands on the tcgen05 tensor cores (TMA-fed, TMEM accumulators), fp32
 * accumulation; D in {64, 128, 256}; ranks and, if asked for, the top-k lists come out of the same epilogue; needs
 * `scratch`; looser parity (operands are rounded to bf16, the target's own column is excluded from the count
 * explicitly).  precision 2: precision 0's RANKS, bit for bit, at tensor-core speed: every fp32 operand
 * is split into two bf16 terms and the tensor cores accumulate hi.hi + hi.lo + lo.hi (K = 3 D); a score farther than
 * eps_r = c_D ||a_r|| max_j ||b_j|| from the row's target (c_64 = 1.5e-4, c_128 = 2e-4, c_256 = 3.1e-4: twice the worst-case sum of
 * the split residual 3.1 2^-16, the fp32 accumulation of 3 D products and the FMA chain's own rounding) decides the
 * comparison as precision 0 would, the pairs inside the band (~0.1 %) are re-scored with precision 0's FMA chain.
 * If the candidate list overflows (degenerate tables) WR_STATUS_EVAL_OVERFLOW is raised: rerun with precision 0.
 * precision 2 with k in [1, 32] (D in {64, 128, 256}, scores_out NULL): precision 0's top-k lists too -- the same ids and
 * the same fp32 values in the same order.  The tensor-core scores pick a per-row candidate set that provably holds the
 * exact top k (every item within 2 eps_r of the running k-th best), and eval_topk_select_kernel re-scores the candidates
 * with precision 0's FMA chain.  `scratch` must then hold wr_eval_scratch_bytes_topk(..., k) bytes.  A row with more than
 * 1,024 candidates is returned with topk_idx[r, 0] = -2 and WR_STATUS_TOPK_OVERFLOW raised: rerun those rows with
 * precision 0 (wr_eval_rank_topk_shard with their target scores); their ranks are already exact.
 */
int wr_eval_rank_topk(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos, int64_t R,
                      int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr, const int32_t *hist_idx,
                      int k, int precision, int32_t *topk_idx, float *topk_val, int32_t *rank, float *target,
                      float *scores_out, void *scratch, void *ws, void *stream);

/* Bytes of 1024-byte-aligned device scratch wr_eval_rank_topk needs for `precision` (0 for precision 0): the bf16
 * copies of the gathered user rows and of the item table that the TMA descriptors point at (three bf16 terms per
 * element for precision 2 -- two for the user rows at D = 256 -- plus its candidate list). */
size_t wr_eval_scratch_bytes(int64_t R, int64_t n_items, int D, int precision);

/* The same for a call that also asks for top-k lists (k = 0: wr_eval_scratch_bytes).  Precision 2 adds a segment of
 * 1,024 candidate item ids and a count per row of a row block (rows are evaluated in blocks of at most 262,144, so the
 * segments stay <= 1 GB); precision 1 needs nothing more. */
size_t wr_eval_scratch_bytes_topk(int64_t R, int64_t n_items, int D, int precision, int k);

/* wr_metrics: BaseRunner.evaluate_method (BaseRunner.py:76-88) from the ranks; float64 means.
 *   hr[i] = mean(rank <= ks[i]);  ndcg[i] = mean((rank <= ks[i]) / log2(rank + 1))
 * host_ks: HOST array of nk cut-offs (nk <= 8); out: DEVICE double [2*nk] = hr[0..nk), ndcg[0..nk).
 */
int wr_metrics(const int32_t *rank, int64_t R, const int *host_ks, int nk, double *out, void *ws, void *stream);

/* ---- row movement for the row-sharded tables (multi-GPU, SURVEY.md section 8e) ---------------------------
 * wr_gather_rows:      out[b] = T[idx[b]]            (owner side of the all-to-all of embedding rows)
 * wr_scatter_add_rows: G[idx[b]] += rows[b]          (owner side of the all-to-all of gradient rows)
 */
int wr_gather_rows(const float *T, const int64_t *idx, int64_t B, int D, int64_t n_rows, float *out, void *ws,
                   void *stream);
int wr_scatter_add_rows(float *G, const int64_t *idx, int64_t B, int D, int64_t n_rows, const float *rows,
                        void *ws, void *stream);

/* ---- negative sampling on the device (SURVEY.md section 8 f-1) --------------------------------------------------
 * wr_neg_sample_mt19937: GeneralModel.Dataset.actions_before_epoch (models/BaseModel.py:167-177) with num_neg = 1,
 * bit-exact on NumPy's global legacy MT19937 stream: the bulk `randint(1, n_items, size=N)` followed, row by row, by
 * scalar redraws while the candidate is in the user's train set.
 *   host_key / pos:   the generator state, `np.random.get_state()[1:3]` (624 words, position 0..624)
 *   user [N]:         int64 user id of every train row, in dataset order;  train_ptr / train_idx: CSR of the sorted
 *                     train_clicked_set per user (int64 [n_users + 1] / int32)
 *   neg_out [N]:      the epoch's negatives (int64)
 *   host_key_out / host_pos_out: the state to hand back to `np.random.set_state` so the host stream continues exactly
 *                     where the reference's would
 * SYNCHRONISES the stream (the state goes back to the host).  Returns WR_E_SIZE if the scratch (sized by
 * wr_neg_sample_scratch_bytes for ~15 % redraws) was too small for this draw: call again with a larger one.
 */
size_t wr_neg_sample_scratch_bytes(int64_t N, int64_t n_items);
int wr_neg_sample_mt19937(const uint32_t *host_key, int pos, int64_t N, const int64_t *user, int64_t n_users,
                          int64_t n_items, const int64_t *train_ptr, const int32_t *train_idx, int64_t *neg_out,
                          uint32_t *host_key_out, int *host_pos_out, void *scratch, size_t scratch_bytes, void *ws,
                          void *stream);

/* wr_pyrandom_sample: HOST function (no GPU): `random.sample(range(n), k)` of CPython's `random` module on its
 * Mersenne Twister state (`random.getstate()[1]`: 624 words + position), bit-exact incl. the state afterwards.  SGL's
 * per-epoch edge dropout (utils/augmentor.py:77-111) is exactly this call on the adjacency's non-zeros. */
int wr_pyrandom_sample(uint32_t *host_state, int *host_pos, int64_t n, int64_t k, int64_t *host_out);

/* ==== one 8 x B200 box: row-sharded tables over NVLink peer memory (SURVEY.md section 8e) =====================
 * One process per GPU.  Every rank owns a slab of device memory (wr_peer_alloc), exports it (wr_peer_export),
 * and maps every other rank's slab (wr_peer_open): after that a kernel on any GPU can load, store and reduce into
 * any rank's rows through NVLink 5 / NVSwitch with ordinary global-memory instructions.  There is no index or row
 * all-to-all: the gather of remote embedding rows and the scatter-add of remote gradient rows happen INSIDE the
 * BPR kernel (ld.global / red.global.add.v4.f32 on peer addresses), the all-gather of a LightGCN layer happens
 * inside the SpMM (neighbour rows are read from their owner), and only the step boundary needs an exchange:
 * wr_peer_barrier.
 *
 * Layout: user u lives on rank u % world at local row u / world; item i on rank i % world at local row
 * rows_u_local + i / world, rows_u_local = ceil(n_users / world).  A rank's shard is therefore one contiguous
 * [rows_u_local + rows_i_local, D] table (P, and M / V / G alike) that its Adam sweep walks with no communication.
 * LightGCN node n is user n if n < n_users, else item n - n_users.
 */
#define WR_MAX_WORLD 8

typedef struct wr_shards {
    float *base[WR_MAX_WORLD]; /* base[g]: rank g's shard as mapped in THIS process (base[rank] is local memory) */
    int32_t world, rank;
    int64_t n_users, n_items;  /* global */
    int64_t rows_u_local;      /* ceil(n_users / world) */
    int64_t rows_i_local;      /* ceil(n_items / world) */
} wr_shards;

int wr_peer_alloc(size_t bytes, void **out_dev_ptr);                 /* cudaMalloc'd, zero-filled, IPC-exportable */
int wr_peer_free(void *dev_ptr);
int wr_peer_export(void *dev_ptr, unsigned char host_handle[64]);    /* cudaIpcGetMemHandle */
int wr_peer_open(const unsigned char host_handle[64], void **out_dev_ptr); /* cudaIpcOpenMemHandle, peer access on */
int wr_peer_close(void *dev_ptr);

/* wr_peer_barrier: all ranks' streams meet.  Everything a rank's stream did before its call (including REDs into
 * peer memory) is visible to every rank's stream after its call.  host_flags[g]: rank g's array of WR_MAX_WORLD
 * uint32 (zeroed once); epoch: 1, 2, 3, ... -- the same on every rank, never reused.
 * If n_values > 0 (<= WR_PEER_VALUES) the barrier doubles as an all-reduce(sum) of that many floats: rank r deposits
 * values_in[0..n) in host_slots[g] on every rank g and, past the barrier, sums_out[v] = sum over ranks, added in
 * rank order (deterministic, identical on every rank).  host_slots[g]: rank g's array of 2 * WR_MAX_WORLD *
 * WR_PEER_VALUES floats (double-buffered by epoch parity).
 * The ranks MUST run on different GPUs (a spin-wait between processes sharing one GPU can deadlock the device).
 * Every cross-GPU wait (here and inside wr_bprmf_step_sharded) gives up after WR_PEER_TIMEOUT_NS and raises
 * WR_STATUS_PEER_TIMEOUT in the workspace status word instead of hanging the GPU when a peer has died.
 */
#define WR_PEER_VALUES 4
int wr_peer_barrier(uint32_t *const host_flags[WR_MAX_WORLD], int world, int rank, uint32_t epoch,
                    float *const host_slots[WR_MAX_WORLD], const float *values_in, int n_values, float *sums_out,
                    void *ws /* nullable: receives WR_STATUS_PEER_TIMEOUT */, void *stream);

/* wr_bpr_fwd_bwd_sharded: wr_bpr_fwd_bwd on this rank's slice of the global batch against sharded tables.
 * T: the embedding shards read (P for BPRMF, the pooled table for LightGCN); Gd: the gradient shards reduced into
 * (remote rows over NVLink).  B: rows in this rank's slice; B_global: rows in the whole batch (the mean and the
 * gradient scale use it).  loss_out[0] = this rank's share, sum_b(loss_b) / B_global -- summed over ranks by
 * wr_peer_barrier it is the batch loss.
 */
int wr_bpr_fwd_bwd_sharded(const wr_shards *host_T, const wr_shards *host_Gd, const int64_t *user,
                           const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global, int D, float gamma,
                           float grad_scale, float *loss_out, void *ws, void *stream);

/* wr_bpr_logsig_sum_fwd_bwd_sharded: wr_bpr_logsig_sum_fwd_bwd (SGL's sum-form BPR) on this rank's slice, with the tables
 * of wr_bpr_fwd_bwd_sharded.  loss_out[0] = this rank's share, sum_b -logsigmoid(s+ - s-) over the slice; the gradient is
 * scaled by grad_scale alone (no 1 / B_global). */
int wr_bpr_logsig_sum_fwd_bwd_sharded(const wr_shards *host_T, const wr_shards *host_Gd, const int64_t *user,
                                      const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global, int D,
                                      float grad_scale, float *loss_out, void *ws, void *stream);

/* wr_infonce_sharded_*: wr_infonce_fwd_bwd for one block (which = 0: the batch's users against all users, 1: the
 * positive items against all items) of row-sharded view tables.  Every rank runs the GLOBAL batch (idx: its B ids, the
 * same on every rank) against ITS OWN rows of the block; the table is never gathered.  Three phases, each rank's calls in
 * this order on its stream, with a wr_peer_barrier between consecutive phases:
 *   partials: gather T1[idx_b] and T2[idx_b] from their owners and normalise them; normalise this rank's real rows of the
 *             block of T2 (padding rows stay out of z); pass 1 against them; this rank's partial z_b is stored into
 *             slot [rank][b] of every rank's z array (host_z[g]: rank g's [world][B] fp32).
 *   weights:  z_b = the world partials summed in rank order (the same bits on every rank); loss_out[0] +=
 *             weight * sum_b (log z_b - a_b . t_{idx_b} / tau) -- the InfoNCE loss of the whole batch, identical on
 *             every rank (add it once, do not sum it over ranks); pass 2 against the local rows, the positive pull by the
 *             owner of idx_b, the table-side chain rule into this rank's rows of dT2; this rank's partial Ga_b ([B, D])
 *             is stored into slot [rank][b] of the owner of idx_b (host_ga[g]: rank g's [world][B][D] fp32, 16-byte
 *             aligned).
 *   batch:    the owner of idx_b sums Ga_b over the ranks in rank order and applies the chain rule through the
 *             normalisation of a_b into its local row of dT1 (RED per occurrence).  No remote loads, no remote REDs.
 * Traffic per block: O(world B D) bytes.  A rank that owns no rows of the block (world > n_users is allowed) takes part in
 * every phase and contributes nothing to z.  D a multiple of 4, at most 256.  scratch: this rank's
 * wr_infonce_sharded_scratch_bytes(B, N_local, D) bytes (N_local: its real rows of the block), the same buffer for the
 * three phases of one block.  Ids outside the block raise WR_STATUS_INDEX_OUT_OF_RANGE and are skipped.
 */
size_t wr_infonce_sharded_scratch_bytes(int64_t B, int64_t N_local, int D);
int wr_infonce_sharded_partials(const wr_shards *host_T1, const wr_shards *host_T2, int which, const int64_t *idx,
                                int64_t B, int D, float tau, float *const host_z[WR_MAX_WORLD], void *scratch,
                                size_t scratch_bytes, void *ws, void *stream);
int wr_infonce_sharded_weights(const wr_shards *host_dT2, int which, const int64_t *idx, int64_t B, int D, float tau,
                               float weight, float grad_scale, float *const host_z[WR_MAX_WORLD],
                               float *const host_ga[WR_MAX_WORLD], float *loss_out, void *scratch, size_t scratch_bytes,
                               void *stream);
int wr_infonce_sharded_batch(const wr_shards *host_dT1, int which, const int64_t *idx, int64_t B, int D, float tau,
                             float weight, float grad_scale, float *const host_ga[WR_MAX_WORLD], void *scratch,
                             size_t scratch_bytes, void *stream);

/* wr_bpr_fwd_bwd_sharded_staged + wr_inbox_scatter: the same for LARGE batches.  16-byte reductions over NVLink do not
 * scale with the number of GPUs (each is its own fabric transaction; measured: 65,536 rows per GPU on 8 GPUs spend
 * 4.5 ms in them), so remote gradient rows are written -- plain coalesced stores -- into the owner's inbox instead, slot
 * 3 b + which of the sender's region (no counters, no atomics), with the owner-local row index + 1 beside them; local
 * rows are still reduced in place.  After the barrier every owner folds its inbox into its gradient shard
 * (wr_inbox_scatter, which also clears the slots).  host_inbox_rows[g] / host_inbox_idx[g]: rank g's
 * [world][cap][D] fp32 / [world][cap] int32 (zero-initialised), cap >= 3 x the largest per-rank batch.
 */
int wr_bpr_fwd_bwd_sharded_staged(const wr_shards *host_T, const wr_shards *host_Gd,
                                  float *const host_inbox_rows[WR_MAX_WORLD], int32_t *const host_inbox_idx[WR_MAX_WORLD],
                                  int64_t cap, const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B,
                                  int64_t B_global, int D, float gamma, float grad_scale, float *loss_out, void *ws,
                                  void *stream);
int wr_inbox_scatter(float *G, const float *inbox_rows, int32_t *inbox_idx, int world, int64_t cap, int D,
                     void *stream);

/* wr_xchg_request / wr_xchg_serve / wr_bpr_fwd_bwd_exchanged: the training step's "all-to-all of indices and embedding
 * rows" (SURVEY.md section 8e) made of posted NVLink stores only.  Loads from peer memory are what does not scale
 * (measured on 8 B200s: random 512-byte row gathers from multi-GB peer mappings reach 30-80 GB/s per GPU -- a TLB miss
 * and a 3.5 us round trip each -- while peer stores stream at link bandwidth), so for batches of >= 8,192 rows per GPU:
 *   wr_xchg_request: every (batch entry, role) of this rank's slice -> owner o, owner-local row r; the entry
 *       (r << 2 | role) is appended to this rank's list in owner o's request array (host_req[o]: rank o's
 *       [world][cap] int32, we write row [rank]; host_req_cnt[o]: rank o's [world] counts) and where[3 b + role] =
 *       o * cap + k remembers the position.  cnt_local: [world] uint32 device scratch, zero on entry, zero on exit.
 *   -- wr_peer_barrier --
 *   wr_xchg_serve: the owner reads every requested row from its LOCAL shard T_local and stores it into the requester's
 *       receive buffer (host_recv[r]: rank r's [world][cap][D] fp32; we write block [rank], in request order).
 *   -- wr_peer_barrier --
 *   wr_bpr_fwd_bwd_exchanged: wr_bpr_fwd_bwd_sharded_staged with the three rows of entry b read from
 *       recv[where[3 b + role]] (local memory); gradient rows go to the owners' inboxes as before.  touched
 *       (nullable): the row map of wr_adam_l2_sweep_marked over this rank's rows -- rows the kernel reduces in place
 *       (entries this rank owns itself) get their bit; wr_inbox_scatter_marked adds the rest.
 * cap >= 3 x the largest per-rank batch.  Ids outside their table raise WR_STATUS_INDEX_OUT_OF_RANGE (entry skipped).
 */
int wr_xchg_request(const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B, int64_t n_users,
                    int64_t n_items, int world, int rank, int32_t *const host_req[WR_MAX_WORLD],
                    uint32_t *const host_req_cnt[WR_MAX_WORLD], int64_t cap, uint32_t *cnt_local, int32_t *where,
                    void *ws, void *stream);
int wr_xchg_serve(const float *T_local, int D, int world, int rank, const int32_t *req_local,
                  const uint32_t *req_cnt_local, int64_t cap, float *const host_recv[WR_MAX_WORLD], void *stream);
int wr_bpr_fwd_bwd_exchanged(const float *recv, const int32_t *where, const wr_shards *host_Gd,
                             float *const host_inbox_rows[WR_MAX_WORLD], int32_t *const host_inbox_idx[WR_MAX_WORLD],
                             int64_t cap, const int64_t *user, const int64_t *pos, const int64_t *neg, int64_t B,
                             int64_t B_global, int D, float gamma, float grad_scale, uint32_t *touched, float *loss_out,
                             void *ws, void *stream);

/* wr_csr_spmm_sharded_dma: wr_csr_spmm_sharded whose output is all-gathered by the COPY ENGINES while the kernel is still
 * running (measured on 8 B200s, 10M x 2M x 494M edges, D = 128: SpMM alone 11.0 ms, with the store-push epilogue 13.8 ms,
 * with the copies beside it 11.6 ms -- the SMs never wait on NVLink).  Rows of Y are counted per block of block_rows
 * (power of two >= 32) as they finish; the warp that completes a block publishes progress flag [block] = epoch, and the
 * side stream holds, per block, one cuStreamWaitValue32 on that flag followed by the world - 1 peer copies of the block
 * (host_push[g] = rank g's copy of this rank's shard of Y, entry [rank] ignored).  `stream` is made to wait for the last
 * copy before the call returns, so the caller's wr_peer_barrier orders the copies before every reader as it does for
 * the store-push form.  progress: DEVICE int32 [progress_words >= 2 ceil(n_local / block_rows)], zero before the first
 * call; epoch: 1, 2, 3, ... per call on the same progress words; nnz: rowptr[n_local] (sizes the two kinds of CTA so
 * that row blocks complete steadily from the start of the kernel; 0 = unknown).  D in {16, 32, 64, 128, 256}.
 * wr_push_shard_dma: the plain all-gather of a finished shard the same way (world - 1 copies on `stream`).
 */
int wr_csr_spmm_sharded_dma(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n_local, int D,
                            const wr_shards *host_X, float *Y, float *add, int zero_add, const float *acc_in,
                            float *acc_out, float acc_div, const wr_spmm_plan *host_plan,
                            float *const host_push[WR_MAX_WORLD], int32_t *progress, int64_t progress_words,
                            int64_t block_rows, uint32_t epoch, int64_t nnz, void *side_stream, void *stream);
int wr_push_shard_dma(const float *src, int64_t n_floats, int world, int rank, float *const host_push[WR_MAX_WORLD],
                      void *stream);

/* wr_push_marked_rows: the all-gather of a row-sharded table that is zero outside a few rows -- the pooled gradient of
 * a batch, input of the first adjoint propagation (LightGCN.py:150-163 backward).  node_bits: bitmap over the GLOBAL node
 * ids [n_users + n_items] (wr_mark_rows on every rank's slice of the batch, OR-ed over the ranks); this rank stores each
 * of ITS rows whose bit is set into host_push[g] + local_row * D for every peer g (host_push[g]: rank g's copy of this
 * rank's shard; entry [rank] ignored).  The unmarked rows of the copies are left as they are: the SpMM that follows
 * gets the same bitmap as wr_spmm_plan.x_rows and never fetches them.  host_X: the table's wr_shards (layout and
 * base[rank] = the local shard).
 */
int wr_push_marked_rows(const wr_shards *host_X, int D, const uint32_t *node_bits, float *const host_push[WR_MAX_WORLD],
                        void *stream);

/* wr_embloss_owner_sumsq / wr_embloss_owner_scatter: EmbLoss (utils/loss.py:83-98, LightGCN.py:165-175) computed by the
 * OWNERS of the ego rows from the request lists of wr_xchg_request, which hold every occurrence of every row of the
 * batch with its role -- no row crosses NVLink:
 *   sumsq_out[0..3) = this rank's sums of squares of the requested user / positive / negative ego rows (the ranks' sums
 *                     meet in wr_peer_barrier);
 *   scatter: G_local[row] += reg_weight / B_global * T_local[row] / sqrt(sumsq_global[role]) per occurrence; if
 *            loss_out != NULL, loss_out[0] += reg_weight * (sum of the three norms) / B_global.
 */
int wr_embloss_owner_sumsq(const float *T_local, int D, int world, const int32_t *req_local,
                           const uint32_t *req_cnt_local, int64_t cap, float *sumsq_out, void *ws, void *stream);
int wr_embloss_owner_scatter(const float *T_local, float *G_local, int D, int world, const int32_t *req_local,
                             const uint32_t *req_cnt_local, int64_t cap, float reg_weight, int64_t B_global,
                             const float *sumsq_global, float *loss_out, void *stream);

/* wr_bprmf_step_sharded: wr_bprmf_step on row-sharded tables -- ONE cooperative launch per rank and step, with the
 * two cross-GPU meeting points inside the kernel: (1) the grid barrier between the BPR phase and the Adam phase is
 * extended across the GPUs by CTA 0 (every rank's remote gradient REDs have landed, the loss shares are exchanged),
 * (2) the last CTA to finish the Adam phase tells every peer that this rank's rows are final, and the next step's
 * kernel waits for that before its first remote gather.  T / Gd: parameter and gradient shards; M / V: this rank's
 * moment shards; epoch: the step number 1, 2, 3, ... (same on every rank, each used once);
 * host_flags[g]: rank g's zero-initialised array of 2 * WR_MAX_WORLD uint32 ([1][r]: rank r's rows are final);
 * host_slots[g]: rank g's zero-initialised, 8-byte aligned array of 2 * WR_MAX_WORLD floats, used as WR_MAX_WORLD 8-byte
 * words: word [r] = {epoch, rank r's loss share} -- arrival and payload in one store, so no fence (an NVLink round trip)
 * sits between them.  loss_out[0] = the loss of the GLOBAL batch (identical on every rank).
 * Supported when wr_bprmf_step_sharded_supported(rows of a shard, D) (cache-sized shards, D in {16,...,256});
 * otherwise use wr_bpr_fwd_bwd_sharded / wr_peer_barrier / wr_adam_l2_sweep / wr_peer_barrier.
 */
int wr_bprmf_step_sharded_supported(int64_t n_local_rows, int D);
int wr_bprmf_step_sharded(const wr_shards *host_T, const wr_shards *host_Gd, float *M, float *V, const int64_t *user,
                          const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global, int D, float gamma,
                          float l2, double beta1, double beta2, float eps, float step_size, float bc2_sqrt,
                          uint32_t epoch, uint32_t *const host_flags[WR_MAX_WORLD],
                          float *const host_slots[WR_MAX_WORLD], float *loss_out, void *ws, void *stream);

/* wr_embloss_sumsq_sharded / wr_embloss_scatter_sharded: the two halves of wr_embloss_fwd_bwd; the three squared
 * norms are batch-global, so the ranks' sums meet (wr_peer_barrier carries them) between the halves.
 *   sumsq_out[0..3)  = this rank's sums of squares of its gathered user / pos / neg ego rows
 *   scatter: g[row] += reg_weight / B_global * row / sqrt(sumsq_global[.]);  if loss_out != NULL,
 *            loss_out[0] += reg_weight * (sum of the three norms) / B_global   (identical on every rank)
 */
int wr_embloss_sumsq_sharded(const wr_shards *host_T, const int64_t *user, const int64_t *pos, const int64_t *neg,
                             int64_t B, int D, float *sumsq_out, void *ws, void *stream);
int wr_embloss_scatter_sharded(const wr_shards *host_T, const wr_shards *host_Gd, const int64_t *user,
                               const int64_t *pos, const int64_t *neg, int64_t B, int64_t B_global, int D,
                               float reg_weight, const float *sumsq_global, float *loss_out, void *ws,
                               void *stream);

/* wr_gather_rows_sharded: out[b] = row idx[b] of the sharded user (which = 0) or item (which = 1) table, read
 * from its owner.  Used by the evaluation to fetch the user rows and the target-item rows of a batch. */
int wr_gather_rows_sharded(const wr_shards *host_T, int which, const int64_t *idx, int64_t B, int D, float *out,
                           void *ws, void *stream);

/* wr_allgather_shards: dst[g] = rank g's shard for every g != rank (dst: local [world, n_local, D] fp32), pulled over
 * NVLink with one streaming kernel.  Together with a wr_shards whose base[g] points at dst[g] (and base[rank] at the own
 * shard) this turns wr_csr_spmm_sharded into "all-gather, then SpMM against a local copy": on power-law graphs the
 * neighbour rows are re-read many times, and only local memory gets those re-reads served by the L2. */
int wr_allgather_shards(const wr_shards *host_src, float *dst, int D, void *stream);

/* wr_csr_spmm_sharded: wr_csr_spmm for this rank's rows of the adjacency (local row l is node l * world + rank of
 * the user block for l < rows_u_local, else of the item block), column ids GLOBAL node ids; X rows are read through
 * host_X -- in place from their owners (small tables), or from a local all-gathered copy (base[g] pointing into it);
 * Y / add / acc_in / acc_out are this rank's local [n_local, D] slabs.
 * host_push (nullable): host_push[g] = where rank g keeps ITS copy of this rank's shard of Y ([n_local, D], peer-mapped;
 * entry [rank] ignored).  Every finished row of Y is then also stored there from the epilogue -- the all-gather of the
 * layer output fused into the SpMM as posted NVLink writes, so the next layer needs no gather pass (measured at 8 GPUs on
 * the 10M x 2M x 494M-edge graph: a separate gather costs as much as the SpMM itself, 10.3 vs 11.1 ms per layer).
 * The caller double-buffers the copies (peers may still be reading the previous layer's) and runs wr_peer_barrier
 * before the next layer reads them.
 */
int wr_csr_spmm_sharded(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n_local, int D,
                        const wr_shards *host_X, float *Y, float *add, int zero_add, const float *acc_in,
                        float *acc_out, float acc_div, const wr_spmm_plan *host_plan,
                        float *const host_push[WR_MAX_WORLD], void *stream);

/* wr_eval_rank_topk_shard: wr_eval_rank_topk against ONE item shard.
 *   Urows   [R, D]  the eval rows' user embeddings, already gathered (wr_gather_rows_sharded)
 *   target  [R]     INPUT: the target scores (wr_rowdot over the gathered rows; precision 1: over bf16-rounded rows)
 *   Iemb    [n_items_local, D] this rank's item rows;  hist_ptr / hist_idx: per USER (indexed by user[r]), holding
 *                   only this shard's items as LOCAL indices, ascending;  pos_local[r]: local index of the target
 *                   if this shard owns it, else -1
 *   rank[r] = 1 + #{local j not in hist : score > target[r]}   =>   global rank = 1 + sum over shards (rank - 1)
 *   topk_idx: LOCAL indices (global item = local * world + shard).
 * D and precision as for wr_eval_rank_topk: D in {16, 32, 64, 128, 256} for precision 0, {64, 128, 256} for 1 and 2.
 * Precision 2 with top-k works here as there (size `scratch` with wr_eval_scratch_bytes_topk over n_items_local; rows
 * marked -2 are rerun with precision 0 on this shard).
 */
int wr_eval_rank_topk_shard(const float *Urows, const float *Iemb, const int64_t *user, const int64_t *pos_local,
                            int64_t R, int64_t n_users, int64_t n_items_local, int D, const int64_t *hist_ptr,
                            const int32_t *hist_idx, int k, int precision, const float *target, int32_t *topk_idx,
                            float *topk_val, int32_t *rank, void *scratch, void *ws, void *stream);

/* wr_rowdot: out[r] = sum_d A[r,d] * B[r,d] as the fp32 FMA chain d = 0..D-1 the scoring kernels use
 * (round_bf16 != 0: operands rounded to bf16 first, as precision 1 does). */
int wr_rowdot(const float *A, const float *B, int64_t R, int D, int round_bf16, float *out, void *stream);

/* wr_topk_merge: final k-way merge of the shards' candidates.  val / idx: [world, R, k] (idx already GLOBAL item
 * ids, unfilled slots -1 / -inf); out: the k best per row, best first, ties to the lower id. */
int wr_topk_merge(const float *val, const int32_t *idx, int world, int64_t R, int k, float *out_val,
                  int32_t *out_idx, void *stream);

/* ---- top-k lists with k up to 256 ---------------------------------------------------------------------------
 * wr_eval_rank_topk_long: wr_eval_rank_topk for 1 <= k <= 256 (lists required, no score dump).  Every row gets precision
 * 0's list: the same item ids in the same order, the same fp32 values (the d = 0 .. D-1 FMA chain), ordered by (value desc,
 * id asc), history items masked, padded with (-1, -inf).  rank and target equal those of a k = 0 call at the same
 * precision.  precision 0: D in {16, 32, 64, 128, 256}; precision 2: D in {64, 128, 256} (tensor cores); precision 1 and
 * any other k: WR_E_TOPK.  The wrappers of this library use it for k > 32 only.
 * Three passes per block of rows: a bound pass takes the k'-th best score of each of n >= S = ceil(k / 32) item ranges
 * (k' = ceil(k / S) <= 32) -- the S-th largest of them, L, bounds the k-th best from below (precision 2: on the
 * tensor-core scores, so the candidates are t >= L - 2 eps_r) -- a collect pass computes the ranks and appends every
 * unmasked item at or above the bound to a 4,096-id segment per row, and a select pass re-scores the candidates with
 * precision 0's FMA chain and sorts them.  A row with more candidates is finished on the device by a sweep over all its items:
 * WR_STATUS_TOPK_OVERFLOW is raised and the 32-bit word at scratch[0] counts those rows; the lists are exact either way.
 * scratch: wr_eval_scratch_bytes_topk_long bytes, 1024-byte aligned (required at both precisions).
 */
int wr_eval_rank_topk_long(const float *Uemb, const float *Iemb, const int64_t *user, const int64_t *pos, int64_t R,
                           int64_t n_users, int64_t n_items, int D, const int64_t *hist_ptr, const int32_t *hist_idx,
                           int k, int precision, int32_t *topk_idx, float *topk_val, int32_t *rank, float *target,
                           void *scratch, void *ws, void *stream);

/* wr_eval_rank_topk_long against ONE item shard, with the arguments of wr_eval_rank_topk_shard (LOCAL list ids). */
int wr_eval_rank_topk_long_shard(const float *Urows, const float *Iemb, const int64_t *user, const int64_t *pos_local,
                                 int64_t R, int64_t n_users, int64_t n_items_local, int D, const int64_t *hist_ptr,
                                 const int32_t *hist_idx, int k, int precision, const float *target, int32_t *topk_idx,
                                 float *topk_val, int32_t *rank, void *scratch, void *ws, void *stream);

/* Bytes of scratch a long call needs (0 for arguments it refuses): the header, precision 2's wr_eval_scratch_bytes, and
 * per row of a block (at most 65,536 rows, so the segments stay <= 1 GB) 16 range bounds, a count and 4,096 ids. */
size_t wr_eval_scratch_bytes_topk_long(int64_t R, int64_t n_items, int D, int precision, int k);

/* wr_topk_merge for lists of 1 <= k <= 256 entries: val / idx [world, R, k]. */
int wr_topk_merge_long(const float *val, const int32_t *idx, int world, int64_t R, int k, float *out_val,
                       int32_t *out_idx, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WHISPRREC_B200_H */
