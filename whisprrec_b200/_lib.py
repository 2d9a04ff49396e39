"""ctypes binding of libwhisprrec_b200.so (the C-ABI declared in include/whisprrec_b200.h).

PyTorch is only the plumbing here: it owns device memory and the stream; every call below hands raw
`data_ptr()`s and the current stream to a hand-written sm_100a kernel.  There is no CPU or eager-torch
fallback: a missing library or a CPU tensor raises.
"""
import ctypes
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libwhisprrec_b200.so')
CSRC = os.path.join(_HERE, 'csrc')

_c = ctypes
_p, _i64, _int, _f32, _sz = _c.c_void_p, _c.c_int64, _c.c_int, _c.c_float, _c.c_size_t
_f64 = _c.c_double

# name -> (restype, argtypes); must list every symbol include/whisprrec_b200.h declares
SIGNATURES = {
    'wr_version': (_int, []),
    'wr_error_string': (_c.c_char_p, [_int]),
    'wr_workspace_bytes': (_sz, []),
    'wr_workspace_init': (_int, [_p, _p]),
    'wr_status': (_int, [_p, _c.POINTER(_c.c_uint32), _p]),
    'wr_bpr_fwd_bwd': (_int, [_p, _p, _p, _p, _p, _i64, _int, _i64, _i64, _f32, _f32, _p, _p, _p, _int, _p, _p]),
    'wr_bpr_logsig_sum_fwd_bwd': (_int, [_p, _p, _p, _p, _p, _i64, _int, _i64, _i64, _f32, _p, _p, _p, _int, _p, _p]),
    'wr_infonce_scratch_bytes': (_sz, [_i64, _i64, _int]),
    'wr_infonce_fwd_bwd': (_int, [_p, _p, _p, _i64, _i64, _int, _f32, _f32, _f32, _p, _p, _p, _p, _sz, _p, _p]),
    'wr_embloss_fwd_bwd': (_int, [_p, _p, _p, _p, _p, _i64, _int, _i64, _i64, _f32, _p, _p, _p, _p, _p]),
    'wr_adam_l2_sweep': (_int, [_p, _p, _p, _p, _i64, _f32, _f64, _f64, _f32, _f32, _f32, _p, _p]),
    'wr_bprmf_step': (_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _i64, _i64, _f32, _f32, _f64, _f64, _f32, _f32,
                             _f32, _p, _p, _p, _p]),
    'wr_bprmf_epoch_scratch_bytes': (_sz, [_i64, _i64]),
    'wr_debug_epoch_trace': (_int, [_p, _p]),
    'wr_debug_step_trace': (_int, [_p]),
    'wr_bprmf_epoch': (_int, [_p, _p, _p, _p, _p, _i64, _i64, _int, _i64, _i64, _f32, _f64, _f32, _f64, _f64, _f32, _i64,
                              _p, _p, _sz, _p, _p]),
    'wr_bprmf_step_host': (_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _i64, _i64, _f32, _f32, _f64, _f64, _f32,
                                  _f32, _f32, _p, _p, _p, _int]),
    'wr_bprmf_ctx_create': (_int, [_p, _p, _p, _p, _i64, _i64, _int, _f32, _f64, _f32, _f64, _f64, _f32, _p, _p,
                                   _c.POINTER(_p)]),
    'wr_bprmf_ctx_step': (_int, [_p, _p, _i64, _i64, _int, _c.POINTER(_f32)]),
    'wr_bprmf_ctx_wait': (_int, [_p, _i64, _int, _c.POINTER(_f32)]),
    'wr_bprmf_ctx_sync': (_int, [_p]),
    'wr_bprmf_ctx_destroy': (_int, [_p]),
    'wr_csr_build_scratch_bytes': (_sz, [_i64]),
    'wr_csr_build': (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _sz, _p, _p]),
    'wr_subgraph_csr_scratch_bytes': (_sz, [_i64]),
    'wr_subgraph_csr': (_int, [_p, _p, _i64, _p, _i64, _int, _p, _p, _p, _p, _sz, _p, _p]),
    'wr_csr_norm_weights': (_int, [_p, _p, _p, _i64, _p, _p]),
    'wr_csr_spmm': (_int, [_p, _p, _p, _i64, _int, _p, _p, _p, _int, _p, _p, _f32, _p, _p]),
    'wr_eval_rank_topk': (_int, [_p, _p, _p, _p, _i64, _i64, _i64, _int, _p, _p, _int, _int, _p, _p, _p, _p, _p, _p,
                                 _p, _p]),
    'wr_eval_scratch_bytes': (_sz, [_i64, _i64, _int, _int]),
    'wr_eval_scratch_bytes_topk': (_sz, [_i64, _i64, _int, _int, _int]),
    'wr_metrics': (_int, [_p, _i64, _c.POINTER(_int), _int, _p, _p, _p]),
    'wr_gather_rows': (_int, [_p, _p, _i64, _int, _i64, _p, _p, _p]),
    'wr_scatter_add_rows': (_int, [_p, _p, _i64, _int, _i64, _p, _p, _p]),
    'wr_neg_sample_scratch_bytes': (_sz, [_i64, _i64]),
    'wr_neg_sample_mt19937': (_int, [_p, _int, _i64, _p, _i64, _i64, _p, _p, _p, _p, _c.POINTER(_int), _p, _sz, _p, _p]),
    'wr_pyrandom_sample': (_int, [_p, _c.POINTER(_int), _i64, _i64, _p]),
    # ---- row-sharded tables over NVLink peer memory ----
    'wr_peer_alloc': (_int, [_sz, _c.POINTER(_p)]),
    'wr_peer_free': (_int, [_p]),
    'wr_peer_export': (_int, [_p, _c.c_char_p]),
    'wr_peer_open': (_int, [_c.c_char_p, _c.POINTER(_p)]),
    'wr_peer_close': (_int, [_p]),
    'wr_peer_barrier': (_int, [_p, _int, _int, _c.c_uint32, _p, _p, _int, _p, _p, _p]),
    'wr_bpr_fwd_bwd_sharded': (_int, [_p, _p, _p, _p, _p, _i64, _i64, _int, _f32, _f32, _p, _p, _p]),
    'wr_bpr_fwd_bwd_sharded_staged': (_int, [_p, _p, _p, _p, _i64, _p, _p, _p, _i64, _i64, _int, _f32, _f32, _p, _p, _p]),
    'wr_xchg_request': (_int, [_p, _p, _p, _i64, _i64, _i64, _int, _int, _p, _p, _i64, _p, _p, _p, _p]),
    'wr_xchg_serve': (_int, [_p, _int, _int, _int, _p, _p, _i64, _p, _p]),
    'wr_bpr_fwd_bwd_exchanged': (_int, [_p, _p, _p, _p, _p, _i64, _p, _p, _p, _i64, _i64, _int, _f32, _f32, _p, _p, _p,
                                        _p]),
    'wr_embloss_owner_sumsq': (_int, [_p, _int, _int, _p, _p, _i64, _p, _p, _p]),
    'wr_embloss_owner_scatter': (_int, [_p, _p, _int, _int, _p, _p, _i64, _f32, _i64, _p, _p, _p]),
    'wr_inbox_scatter': (_int, [_p, _p, _p, _int, _i64, _int, _p]),
    'wr_csr_spmm_sharded_dma': (_int, [_p, _p, _p, _i64, _int, _p, _p, _p, _int, _p, _p, _f32, _p, _p, _p, _i64, _i64,
                                       _c.c_uint32, _i64, _p, _p]),
    'wr_push_shard_dma': (_int, [_p, _i64, _int, _int, _p, _p]),
    'wr_push_marked_rows': (_int, [_p, _int, _p, _p, _p]),
    'wr_inbox_scatter_marked': (_int, [_p, _p, _p, _int, _i64, _int, _p, _p]),
    'wr_mark_rows': (_int, [_p, _p, _p, _i64, _i64, _i64, _p, _p]),
    'wr_adam_l2_sweep_marked': (_int, [_p, _p, _p, _p, _i64, _int, _p, _f32, _f64, _f64, _f32, _f32, _f32, _p, _p]),
    'wr_bprmf_step_marked': (_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _int, _i64, _i64, _f32, _f32, _f64, _f64, _f32,
                                    _f32, _f32, _p, _p, _p, _p]),
    'wr_bprmf_step_sharded_supported': (_int, [_i64, _int]),
    'wr_bprmf_step_sharded': (_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, _int, _f32, _f32, _f64, _f64, _f32, _f32,
                                     _f32, _c.c_uint32, _p, _p, _p, _p, _p]),
    'wr_embloss_sumsq_sharded': (_int, [_p, _p, _p, _p, _i64, _int, _p, _p, _p]),
    'wr_embloss_scatter_sharded': (_int, [_p, _p, _p, _p, _p, _i64, _i64, _int, _f32, _p, _p, _p, _p]),
    'wr_gather_rows_sharded': (_int, [_p, _int, _p, _i64, _int, _p, _p, _p]),
    'wr_allgather_shards': (_int, [_p, _p, _int, _p]),
    'wr_csr_spmm_sharded': (_int, [_p, _p, _p, _i64, _int, _p, _p, _p, _int, _p, _p, _f32, _p, _p, _p]),
    'wr_eval_rank_topk_shard': (_int, [_p, _p, _p, _p, _i64, _i64, _i64, _int, _p, _p, _int, _int, _p, _p, _p, _p,
                                       _p, _p, _p]),
    'wr_rowdot': (_int, [_p, _p, _i64, _int, _int, _p, _p]),
    'wr_topk_merge': (_int, [_p, _p, _int, _i64, _int, _p, _p, _p]),
    # ---- top-k lists of up to 256 items ----
    'wr_eval_rank_topk_long': (_int, [_p, _p, _p, _p, _i64, _i64, _i64, _int, _p, _p, _int, _int, _p, _p, _p, _p, _p,
                                      _p, _p]),
    'wr_eval_rank_topk_long_shard': (_int, [_p, _p, _p, _p, _i64, _i64, _i64, _int, _p, _p, _int, _int, _p, _p, _p, _p,
                                            _p, _p, _p]),
    'wr_eval_scratch_bytes_topk_long': (_sz, [_i64, _i64, _int, _int, _int]),
    'wr_topk_merge_long': (_int, [_p, _p, _int, _i64, _int, _p, _p, _p]),
}

_lib = None


class WhisprError(RuntimeError):
    pass


def build(verbose=False):
    """Compile the library in-tree with nvcc for sm_100a (works without a GPU)."""
    r = subprocess.run(['make', '-C', CSRC, '-j4'], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode != 0:
        raise WhisprError('building libwhisprrec_b200.so failed')
    return LIB_PATH


def load():
    """dlopen the library and attach signatures.  Raises (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise WhisprError(f'{LIB_PATH} not found: run `python -c "import __graft_entry__ as g; g.build()"` '
                              f'or `make -C {CSRC}`; there is no CPU fallback')
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.wr_version() != 100:
            raise WhisprError('libwhisprrec_b200.so version mismatch')
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise WhisprError(f'whisprrec_b200 error {rc}: {load().wr_error_string(rc).decode()}')


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise WhisprError('whisprrec_b200 kernels need CUDA tensors (no CPU fallback)')
    if dtype is not None and t.dtype != dtype:
        raise WhisprError(f'expected {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise WhisprError('tensor must be contiguous')
    return t.data_ptr()


class Workspace:
    """Device scratch for the reductions; one per stream."""

    def __init__(self, device):
        lib = load()
        self.buf = torch.empty(lib.wr_workspace_bytes(), dtype=torch.uint8, device=device)
        check(lib.wr_workspace_init(self.buf.data_ptr(), stream_ptr()))
        # rows of the last top-k call that were rerun at precision 0 (k <= 32) or finished by the row sweep (k > 32)
        self.last_topk_fallback_rows = 0

    @property
    def ptr(self):
        return self.buf.data_ptr()

    def status(self):
        """Read-and-clear the device status word (synchronises)."""
        out = ctypes.c_uint32(0)
        check(load().wr_status(self.ptr, ctypes.byref(out), stream_ptr()))
        return out.value

    def restore_status(self, bits):
        """OR `bits` back into the device status word (after a caller has read-and-cleared it for its own bit)."""
        self.buf[:4].view(torch.int32).bitwise_or_(int(bits))

    def raise_on_status(self):
        st = self.status()
        if st & 2:
            raise WhisprError('a cross-GPU wait timed out: a peer rank died or fell out of step')
        if st & 1:
            raise IndexError('index out of range in self')      # what nn.Embedding raises in the reference


# ------------------------------------------------------------------------------------------------------
# thin tensor-level wrappers (argument checks live in the C side)
# ------------------------------------------------------------------------------------------------------
F32, I64, I32 = torch.float32, torch.int64, torch.int32


def bpr_fwd_bwd(U, I, user, pos, neg, gU, gI, loss_out, ws, gamma=1e-10, grad_scale=1.0, accumulate_loss=False):
    D = U.shape[1]
    check(load().wr_bpr_fwd_bwd(ptr(U, F32), ptr(I, F32), ptr(user, I64), ptr(pos, I64), ptr(neg, I64),
                                user.numel(), D, U.shape[0], I.shape[0], gamma, grad_scale,
                                ptr(gU, F32), ptr(gI, F32), ptr(loss_out, F32), int(accumulate_loss),
                                ws.ptr, stream_ptr()))


def bpr_logsig_sum_fwd_bwd(U, I, user, pos, neg, gU, gI, loss_out, ws, grad_scale=1.0, accumulate_loss=False):
    """SGL's BPR term: sum_b -logsigmoid(s+ - s-) (SGL.py:176-185)."""
    check(load().wr_bpr_logsig_sum_fwd_bwd(ptr(U, F32), ptr(I, F32), ptr(user, I64), ptr(pos, I64), ptr(neg, I64),
                                           user.numel(), U.shape[1], U.shape[0], I.shape[0], grad_scale, ptr(gU, F32),
                                           ptr(gI, F32), ptr(loss_out, F32), int(accumulate_loss), ws.ptr, stream_ptr()))


def infonce_fwd_bwd(T1, T2, idx, tau, weight, grad_scale, dT1, dT2, loss_out, ws, scratch=None):
    """InfoNCE of SGL.py:196-231 for one block of rows, forward + backward (wr_infonce_fwd_bwd); returns the scratch
    tensor so that the caller can hand it back next time."""
    B, (N, D) = idx.numel(), T2.shape
    nbytes = load().wr_infonce_scratch_bytes(B, N, D)
    if scratch is None or scratch.numel() < nbytes:
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=T1.device)
    check(load().wr_infonce_fwd_bwd(ptr(T1, F32), ptr(T2, F32), ptr(idx, I64), B, N, D, tau, weight, grad_scale,
                                    ptr(dT1, F32), ptr(dT2, F32), ptr(loss_out, F32), scratch.data_ptr(), scratch.numel(),
                                    ws.ptr, stream_ptr()))
    return scratch


def embloss_fwd_bwd(U0, I0, user, pos, neg, gU0, gI0, loss_out, ws, reg_weight):
    D = U0.shape[1]
    check(load().wr_embloss_fwd_bwd(ptr(U0, F32), ptr(I0, F32), ptr(user, I64), ptr(pos, I64), ptr(neg, I64),
                                    user.numel(), D, U0.shape[0], I0.shape[0], reg_weight,
                                    ptr(gU0, F32), ptr(gI0, F32), ptr(loss_out, F32), ws.ptr, stream_ptr()))


def adam_scalars(step, lr, beta1=0.9, beta2=0.999):
    """(lr / (1 - beta1^t), sqrt(1 - beta2^t)) in Python doubles, as torch/optim/adam.py computes them."""
    return lr / (1.0 - beta1 ** step), (1.0 - beta2 ** step) ** 0.5


def adam_l2_sweep(P, M, V, G, step, lr, l2, beta1=0.9, beta2=0.999, eps=1e-8, dev_scalars=None):
    ss, bc2s = adam_scalars(step, lr, beta1, beta2)
    check(load().wr_adam_l2_sweep(ptr(P, F32), ptr(M, F32), ptr(V, F32), ptr(G, F32), P.numel(), l2, beta1, beta2,
                                  eps, ss, bc2s, ptr(dev_scalars, F32), stream_ptr()))


FUSED_STEP_MAX_ELEMS = 8 << 20      # WR_FUSED_STEP_MAX_ELEMS of csrc/train_kernels.cu: beyond it steps stream from HBM


def row_map(n_rows, device):
    """The `touched` bitmap of the row-marked entry points: one bit per table row, all zero between steps."""
    return torch.zeros((n_rows + 31) // 32, dtype=I32, device=device)


def adam_l2_sweep_marked(P, M, V, G, touched, step, lr, l2, beta1=0.9, beta2=0.999, eps=1e-8, dev_scalars=None):
    """adam_l2_sweep for a gradient that is zero outside the rows whose bit is set in `touched` (cleared on return)."""
    if touched.numel() < (P.shape[0] + 31) // 32:
        raise WhisprError('row map too small for the table')
    ss, bc2s = adam_scalars(step, lr, beta1, beta2)
    check(load().wr_adam_l2_sweep_marked(ptr(P, F32), ptr(M, F32), ptr(V, F32), ptr(G, F32), P.shape[0], P.shape[1],
                                         ptr(touched, I32), l2, beta1, beta2, eps, ss, bc2s, ptr(dev_scalars, F32),
                                         stream_ptr()))


def mark_rows(user, pos, neg, n_users, n_items, touched):
    if touched.numel() < (n_users + n_items + 31) // 32:
        raise WhisprError('row map too small for the table')
    check(load().wr_mark_rows(ptr(user, I64), ptr(pos, I64), ptr(neg, I64), user.numel(), n_users, n_items,
                              ptr(touched, I32), stream_ptr()))


def bprmf_step(P, M, V, G, user, pos, neg, n_users, step, lr, l2, loss_out, ws, beta1=0.9, beta2=0.999, eps=1e-8,
               gamma=1e-10, dev_scalars=None, touched=None):
    """One BPRMF iteration (zero_grad + predict + backward + Adam.step) on the fused tables.  With a row map
    (`touched`, see row_map) tables beyond the caches skip the gradient rows the batch did not touch."""
    ss, bc2s = adam_scalars(step, lr, beta1, beta2)
    if touched is not None:
        if touched.numel() < (P.shape[0] + 31) // 32:
            raise WhisprError('row map too small for the table')
        check(load().wr_bprmf_step_marked(ptr(P, F32), ptr(M, F32), ptr(V, F32), ptr(G, F32), ptr(touched, I32),
                                          ptr(user, I64), ptr(pos, I64), ptr(neg, I64), user.numel(), P.shape[1], n_users,
                                          P.shape[0] - n_users, gamma, l2, beta1, beta2, eps, ss, bc2s,
                                          ptr(dev_scalars, F32), ptr(loss_out, F32), ws.ptr, stream_ptr()))
        return
    check(load().wr_bprmf_step(ptr(P, F32), ptr(M, F32), ptr(V, F32), ptr(G, F32), ptr(user, I64), ptr(pos, I64),
                               ptr(neg, I64), user.numel(), P.shape[1], n_users, P.shape[0] - n_users, gamma, l2,
                               beta1, beta2, eps, ss, bc2s, ptr(dev_scalars, F32), ptr(loss_out, F32), ws.ptr,
                               stream_ptr()))


def bprmf_epoch(P, M, V, G, ids, batch, n_users, adam_t0, lr, l2, losses, ws, beta1=0.9, beta2=0.999, eps=1e-8,
                gamma=1e-10, resident=True):
    """Every step of an epoch from one call; ids: contiguous int64 [3, N] device tensor in batch order.  Tables that
    fit the SMs' shared memory run as ONE resident launch (resident=False forces one launch per step)."""
    N = ids.shape[1]
    if ids.dim() != 2 or ids.shape[0] != 3 or losses.numel() < (N + batch - 1) // batch:
        raise WhisprError('ids must be [3, N] and losses hold one float per step')
    lib = load()
    nbytes = lib.wr_bprmf_epoch_scratch_bytes(N, batch) if resident else 0
    scratch = torch.empty(nbytes // 16 * 2 + 2, dtype=torch.int64, device=P.device) if nbytes else None   # 16 B aligned
    check(lib.wr_bprmf_epoch(ptr(P, F32), ptr(M, F32), ptr(V, F32), ptr(G, F32), ptr(ids, I64), N, batch, P.shape[1],
                             n_users, P.shape[0] - n_users, gamma, lr, l2, beta1, beta2, eps, adam_t0,
                             ptr(losses, F32), None if scratch is None else scratch.data_ptr(), nbytes, ws.ptr,
                             stream_ptr()))
    return (N + batch - 1) // batch


def bprmf_step_host(host_ids, dev_ids, host_loss, P, M, V, G, n_users, step, lr, l2, loss_out, ws, beta1=0.9,
                    beta2=0.999, eps=1e-8, gamma=1e-10, sync=True):
    """The same iteration from pinned host ids [3, B]; the batch loss lands in the pinned `host_loss`."""
    if host_ids.is_cuda or not host_ids.is_pinned() or not host_loss.is_pinned():
        raise WhisprError('host_ids / host_loss must be pinned host tensors')
    if host_ids.dtype != I64 or host_ids.dim() != 2 or host_ids.shape[0] != 3 or not host_ids.is_contiguous():
        raise WhisprError('host_ids must be a contiguous int64 [3, B] tensor')
    B = host_ids.shape[1]
    if dev_ids.numel() < 3 * B:
        raise WhisprError('device staging too small')
    ss, bc2s = adam_scalars(step, lr, beta1, beta2)
    check(load().wr_bprmf_step_host(host_ids.data_ptr(), ptr(dev_ids, I64), host_loss.data_ptr(), ptr(P, F32),
                                    ptr(M, F32), ptr(V, F32), ptr(G, F32), B, P.shape[1], n_users,
                                    P.shape[0] - n_users, gamma, l2, beta1, beta2, eps, ss, bc2s, ptr(loss_out, F32),
                                    ws.ptr, stream_ptr(), int(sync)))


class BprmfContext:
    """wr_bprmf_ctx: host-fed BPRMF training on the resident kernel (pinned or pageable ids in, loss out)."""

    def __init__(self, P, M, V, G, n_users, lr, l2, ws, beta1=0.9, beta2=0.999, eps=1e-8, gamma=1e-10):
        self._keep = (P, M, V, G, ws)
        self._h = _p()
        self._loss = _f32(0.0)
        lib = load()
        self._step, self._wait = lib.wr_bprmf_ctx_step, lib.wr_bprmf_ctx_wait
        self.steps = 0
        check(lib.wr_bprmf_ctx_create(ptr(P, F32), ptr(M, F32), ptr(V, F32), ptr(G, F32), n_users,
                                      P.shape[0] - n_users, P.shape[1], gamma, lr, l2, beta1, beta2, eps, ws.ptr,
                                      stream_ptr(), ctypes.byref(self._h)))

    def step(self, host_ids_ptr, B, adam_t, wait=1):
        """host_ids_ptr: address of a [3, B] int64 host buffer.  wait: 1 = until the step is complete, 2 = until the
        loss is out (the Adam phase may still be running), 0 = not at all (collect with wait()).  Returns the batch
        loss (float; meaningless for wait=0)."""
        rc = self._step(self._h, host_ids_ptr, B, adam_t, int(wait), ctypes.byref(self._loss))
        if rc:
            check(rc)
        self.steps += 1
        return self._loss.value

    def wait(self, step, wait=1):
        """Loss of the context's `step`-th step (0-based), once it is complete (1) / its loss is out (2)."""
        rc = self._wait(self._h, step, int(wait), ctypes.byref(self._loss))
        if rc:
            check(rc)
        return self._loss.value

    def sync(self):
        """Close the resident kernel: M / V are back in global memory and the caller's stream is ordered behind it."""
        if self._h:
            check(load().wr_bprmf_ctx_sync(self._h))

    def close(self):
        if self._h:
            load().wr_bprmf_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass


def csr_build(users, items, n_users, n_items, ws):
    """wr_csr_build: (user, item) int64 device tensors -> (rowptr int64 [N + 1], col int32 [nnz]) of the bipartite
    adjacency, rows and columns ascending, duplicate pairs dropped.  Synchronises once (nnz comes back to the host)."""
    E = users.numel()
    if items.numel() != E:
        raise WhisprError('users / items must have the same length')
    dev = users.device
    N = int(n_users) + int(n_items)
    lib = load()
    rowptr = torch.empty(N + 1, dtype=I64, device=dev)
    col = torch.empty(2 * E, dtype=I32, device=dev)
    nnz = torch.zeros(1, dtype=I64, device=dev)
    nbytes = lib.wr_csr_build_scratch_bytes(E)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    check(lib.wr_csr_build(ptr(users, I64), ptr(items, I64), E, n_users, n_items, ptr(rowptr, I64), ptr(col, I32),
                           ptr(nnz, I64), scratch.data_ptr(), nbytes, ws.ptr, stream_ptr()))
    n = int(nnz.item())
    del scratch
    return rowptr, col[:n]


def subgraph_csr(rowptr, col, keep, ws, transpose=False):
    """wr_subgraph_csr: (rowptr int64 [N + 1], col int32 [kept]) of the sub-graph keeping edges `keep` (int64 device tensor
    of edge numbers in CSR order) of the square CSR matrix (rowptr, col), or of its transpose."""
    K, N = keep.numel(), rowptr.numel() - 1
    dev = keep.device
    lib = load()
    out_ptr = torch.empty(N + 1, dtype=I64, device=dev)
    out_col = torch.empty(K, dtype=I32, device=dev)
    nnz = torch.zeros(1, dtype=I64, device=dev)
    nbytes = lib.wr_subgraph_csr_scratch_bytes(K)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    check(lib.wr_subgraph_csr(ptr(rowptr, I64), ptr(col, I32), N, ptr(keep, I64), K, int(transpose), ptr(out_ptr, I64),
                              ptr(out_col, I32), ptr(nnz, I64), scratch.data_ptr(), nbytes, ws.ptr, stream_ptr()))
    return out_ptr, out_col[:int(nnz.item())]


def csr_norm_weights(rowptr, col, dinv, val):
    check(load().wr_csr_norm_weights(ptr(rowptr, I64), ptr(col, I32), ptr(dinv, F32), rowptr.numel() - 1,
                                     ptr(val, F32), stream_ptr()))


class _PlanStruct(ctypes.Structure):
    """Mirror of `wr_spmm_plan` (include/whisprrec_b200.h)."""
    _fields_ = [('long_threshold', _i64), ('n_chunks', _i64), ('n_long', _i64),
                ('chunk_row', _p), ('chunk_beg', _p), ('chunk_len', _p), ('chunk_slot', _p), ('slot_chunks', _p),
                ('slot_arrivals', _p), ('slot_partial', _p), ('hot_bits', _p), ('x_rows', _p)]


def _plan_ref(plan, x_rows, keep):
    """Pointer to the wr_spmm_plan of a call: the plan's own struct, or a copy of it carrying the per-call x_rows map."""
    base = None if plan is None else plan.struct
    if x_rows is None:
        return None if base is None else ctypes.addressof(base)
    st = _PlanStruct()
    if base is not None:
        ctypes.memmove(ctypes.addressof(st), ctypes.addressof(base), ctypes.sizeof(st))
    else:
        st.long_threshold = (1 << 63) - 1
    st.x_rows = ptr(x_rows, I32)
    keep.append(st)
    return ctypes.addressof(st)


class SpmmPlan:
    """Slices of the rows with more than `threshold` non-zeros, so that no warp walks more than `chunk` edges.

    Built once per graph from the host row pointers (vectorised NumPy, O(rows)); the device arrays and the
    zeroed scratch live as long as the plan does.
    """

    def __init__(self, rowptr_host, D, device, threshold=128, chunk=128, hot_budget_bytes=0,
                 hot_min_table_bytes=96 << 20):
        import numpy as np
        deg = np.diff(rowptr_host)
        long_rows = np.nonzero(deg > threshold)[0]
        self.threshold, self.chunk, self.n_long = int(threshold), int(chunk), int(len(long_rows))
        per_row = (deg[long_rows] + chunk - 1) // chunk
        self.n_chunks = int(per_row.sum())
        self.struct = None
        # optional (off by default: measured a 5 % LOSS at 10M x 2M x 494M edges, profiles/r02_spmm_hot_rows.json -- the
        # 80 MB hottest rows carry only 31 % of the reads and the bitmap test costs more than the hits save): the
        # highest-degree nodes (the adjacency is symmetric: a node's column is read once per edge of its row) get their
        # rows loaded with an L2 evict_last policy, as many as fit in the budget
        self.hot_bits, self.n_hot = None, 0
        n = len(deg)
        if hot_budget_bytes and n * D * 4 > hot_min_table_bytes:
            k = min(n, int(hot_budget_bytes) // (D * 4))
            if k > 0:
                thr = np.partition(deg, n - k)[n - k]
                hot = deg > thr
                room = k - int(hot.sum())
                if room > 0:
                    ties = np.nonzero(deg == thr)[0][:room]
                    hot[ties] = True
                self.n_hot = int(hot.sum())
                bits = np.packbits(np.pad(hot, (0, (-n) % 32)), bitorder='little').view(np.uint32)
                self.hot_bits = torch.from_numpy(np.ascontiguousarray(bits).view(np.int32)).to(device)
        if self.n_chunks == 0 and self.hot_bits is None:
            return
        to = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a.astype(dt))).to(device)
        if self.n_chunks:
            slot = np.repeat(np.arange(self.n_long, dtype=np.int32), per_row)
            first = np.zeros(self.n_long, dtype=np.int64)
            np.cumsum(per_row[:-1], out=first[1:])
            k = np.arange(self.n_chunks, dtype=np.int64) - first[slot]          # slice number inside its row
            beg = rowptr_host[long_rows][slot] + k * chunk
            length = np.minimum(chunk, rowptr_host[long_rows + 1][slot] - beg)
            self.chunk_row, self.chunk_beg = to(long_rows[slot], np.int32), to(beg, np.int64)
            self.chunk_len, self.chunk_slot = to(length, np.int32), to(slot, np.int32)
            self.slot_chunks = to(per_row, np.int32)
            self.slot_arrivals = torch.zeros(self.n_long, dtype=I32, device=device)
            self.slot_partial = torch.zeros((self.n_long, D), dtype=F32, device=device)
            self.struct = _PlanStruct(self.threshold, self.n_chunks, self.n_long, self.chunk_row.data_ptr(),
                                      self.chunk_beg.data_ptr(), self.chunk_len.data_ptr(), self.chunk_slot.data_ptr(),
                                      self.slot_chunks.data_ptr(), self.slot_arrivals.data_ptr(),
                                      self.slot_partial.data_ptr(), None)
        else:
            self.struct = _PlanStruct(self.threshold, 0, 0, None, None, None, None, None, None, None, None)
        if self.hot_bits is not None:
            self.struct.hot_bits = self.hot_bits.data_ptr()

    def ref(self):
        return None if self.struct is None else ctypes.addressof(self.struct)


def csr_spmm(rowptr, col, val, X, Y=None, add=None, zero_add=False, acc_in=None, acc_out=None, acc_div=1.0,
             plan=None, x_rows=None):
    """x_rows: optional bitmap over the rows of X (row_map): rows whose bit is clear are zero and are not fetched."""
    N, D = X.shape
    if x_rows is not None and x_rows.numel() < (N + 31) // 32:
        raise WhisprError('row map too small for X')
    keep = []
    check(load().wr_csr_spmm(ptr(rowptr, I64), ptr(col, I32), ptr(val, F32), N, D, ptr(X, F32), ptr(Y, F32),
                             ptr(add, F32), int(zero_add), ptr(acc_in, F32), ptr(acc_out, F32), acc_div,
                             _plan_ref(plan, x_rows, keep), stream_ptr()))


def exact_tc_supported(D, k=0, scores=False):
    """The ranks-only predicate: precision 2 (precision 0's ranks on the tensor cores) covers D in {64, 128, 256} for
    calls without top-k lists or a score dump.  Calls with lists: exact_tc_topk_supported."""
    return D in (64, 128, 256) and k == 0 and not scores


def exact_tc_topk_supported(D, k, scores=False):
    """precision 2 with top-k lists (precision 0's lists on the tensor cores): D in {64, 128, 256}, 1 <= k <= 32, no
    score dump."""
    return D in (64, 128, 256) and 1 <= k <= 32 and not scores


TOPK_KMAX = 32             # lists of wr_eval_rank_topk
TOPK_LONG_KMAX = 256       # lists of wr_eval_rank_topk_long


def exact_tc_topk_long_supported(D, k):
    """precision 2 with long lists (wr_eval_rank_topk_long on the tensor cores): D in {64, 128, 256}, 1 <= k <= 256.
    The wrappers below use that entry point for k > 32 only."""
    return D in (64, 128, 256) and 1 <= k <= TOPK_LONG_KMAX


def _long_precision(D, k, precision, scores):
    """The precision a list of k > 32 items is computed at: 2 on the tensor cores where they cover D, else 0."""
    if precision == 1:
        raise WhisprError(f'precision 1 gives top-k lists of at most {TOPK_KMAX} items (k = {k}); use precision 0 or 2')
    if scores:
        raise WhisprError(f'no dense score dump with top-k lists of more than {TOPK_KMAX} items')
    if k > TOPK_LONG_KMAX:
        raise WhisprError(f'top-k lists hold at most {TOPK_LONG_KMAX} items (k = {k})')
    return 2 if precision == 2 and exact_tc_topk_long_supported(D, k) else 0


def _aligned_scratch(nbytes, dev):
    scratch = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
    off = (-scratch.data_ptr()) % 1024
    return scratch[off:off + nbytes]


def _long_call(launch, R, n_items, D, k, precision, ws):
    """One wr_eval_rank_topk_long(_shard) call, launch(precision, scratch_ptr).  Precision 2 whose rank candidate list
    overflowed (degenerate tables) is repeated at precision 0.  Rows finished by the device-side sweep go to
    ws.last_topk_fallback_rows; status bits that are not the call's own are handed back."""
    keep = 0
    for p in ((2, 0) if precision == 2 else (0,)):
        scratch = _aligned_scratch(load().wr_eval_scratch_bytes_topk_long(R, n_items, D, p, k), ws.buf.device)
        out = launch(p, scratch.data_ptr())
        st = ws.status()
        keep |= st & ~12
        if not (p == 2 and st & 4):
            break
    ws.last_topk_fallback_rows = int(scratch[:4].view(torch.int32).item())
    if keep:
        ws.restore_status(keep)
    return out


def _eval_rank_topk_long(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k, precision):
    R, D = user.numel(), Uemb.shape[1]
    dev = Uemb.device
    rank = torch.empty(R, dtype=I32, device=dev)
    target = torch.empty(R, dtype=F32, device=dev)
    tki = torch.empty((R, k), dtype=I32, device=dev)
    tkv = torch.empty((R, k), dtype=F32, device=dev)

    def launch(p, scratch):
        check(load().wr_eval_rank_topk_long(ptr(Uemb, F32), ptr(Iemb, F32), ptr(user, I64), ptr(pos, I64), R,
                                            Uemb.shape[0], Iemb.shape[0], D, ptr(hist_ptr, I64), ptr(hist_idx, I32), k,
                                            p, ptr(tki, I32), ptr(tkv, F32), ptr(rank, I32), ptr(target, F32), scratch,
                                            ws.ptr, stream_ptr()))
        return rank, target, tki, tkv, None
    return _long_call(launch, R, Iemb.shape[0], D, k, precision, ws)


def _eval_rank_topk_long_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k, precision):
    R, D = user.numel(), Urows.shape[1]
    dev = Urows.device
    rank = torch.empty(R, dtype=I32, device=dev)
    tki = torch.empty((R, k), dtype=I32, device=dev)
    tkv = torch.empty((R, k), dtype=F32, device=dev)

    def launch(p, scratch):
        check(load().wr_eval_rank_topk_long_shard(ptr(Urows, F32), ptr(Iemb, F32), ptr(user, I64), ptr(pos_local, I64),
                                                  R, n_users, Iemb.shape[0], D, ptr(hist_ptr, I64), ptr(hist_idx, I32),
                                                  k, p, ptr(target, F32), ptr(tki, I32), ptr(tkv, F32), ptr(rank, I32),
                                                  scratch, ws.ptr, stream_ptr()))
        return rank, tki, tkv
    return _long_call(launch, R, Iemb.shape[0], D, k, precision, ws)


def _exact_topk_fallback(out, U, gathered, Iemb, user, pos, n_users, hist_ptr, hist_idx, target, ws, k):
    """Rows of a precision-2 top-k call whose candidate segment overflowed (topk_idx[r, 0] = -2): their lists again with
    precision 0, on those rows only (item-shard mode with their targets); the ranks are exact already.  U: the user
    table (gathered = False) or one row per eval row (gathered = True)."""
    tki, tkv = out[-2], out[-1]
    bad = (tki[:, 0] == -2).nonzero().flatten()
    ws.last_topk_fallback_rows = bad.numel()
    if bad.numel():
        rows = U.index_select(0, bad) if gathered else gather_rows(U, user[bad].contiguous(), ws)
        _, bi, bv = _eval_rank_topk_shard(rows.contiguous(), Iemb, user[bad].contiguous(), pos[bad].contiguous(),
                                          n_users, hist_ptr, hist_idx, target[bad].contiguous(), ws, k, 0)
        tki[bad] = bi
        tkv[bad] = bv


def eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k=0, precision=0, scores=False):
    """Returns (rank int32 [R], target fp32 [R], topk_idx int32 [R,k] | None, topk_val fp32 [R,k] | None,
    scores fp32 [R, n_items] | None).  precision: 0 fp32 FMA tiles; 1 bf16 tensor cores; 2 split-bf16 tensor cores +
    exact re-check (ranks identical to 0; if the candidate list overflows -- degenerate tables -- the call is repeated
    with precision 0, which costs one synchronisation).  Precision 2 with k in 1..32 gives precision 0's lists too: rows
    whose list candidates overflow their segment are rerun alone at precision 0 (ws.last_topk_fallback_rows).
    k in 33..256 (precision 0 or 2; 2 falls back to 0 where the tensor cores do not cover D): the same lists from
    wr_eval_rank_topk_long; rows with more candidates than their segment holds are finished on the device
    (ws.last_topk_fallback_rows)."""
    R, D = user.numel(), Uemb.shape[1]
    if k > TOPK_KMAX:
        return _eval_rank_topk_long(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k,
                                    _long_precision(D, k, precision, scores))
    if precision == 2 and k > 0:
        if not exact_tc_topk_supported(D, k, scores):
            return _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k, 0, scores)
        out = _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k, 2, False)
        st = ws.status()
        ws.last_topk_fallback_rows = 0
        if st & 4:
            out = _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k, 0, False)
            ws.last_topk_fallback_rows = R
        elif st & 8:
            _exact_topk_fallback(out[2:4], Uemb, False, Iemb, user, pos, Uemb.shape[0], hist_ptr, hist_idx, out[1], ws, k)
        st &= ~12
        if st:
            ws.restore_status(st)
        return out
    if precision == 2:
        if not exact_tc_supported(D, k, scores):
            precision = 0
        else:
            out = _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, 0, 2, False)
            st = ws.status()
            if st & 4:
                out = _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, 0, 0, False)
                st &= ~4
            if st:                       # hand the other bits back to the caller's raise_on_status
                ws.restore_status(st)
            return out
    return _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k, precision, scores)


def _eval_rank_topk(Uemb, Iemb, user, pos, hist_ptr, hist_idx, ws, k, precision, scores):
    R, D = user.numel(), Uemb.shape[1]
    dev = Uemb.device
    rank = torch.empty(R, dtype=I32, device=dev)
    target = torch.empty(R, dtype=F32, device=dev)
    tki = torch.empty((R, k), dtype=I32, device=dev) if k > 0 else None
    tkv = torch.empty((R, k), dtype=F32, device=dev) if k > 0 else None
    sc = torch.empty((R, Iemb.shape[0]), dtype=F32, device=dev) if scores else None
    nbytes = load().wr_eval_scratch_bytes_topk(R, Iemb.shape[0], D, precision, k)
    scratch = None
    if nbytes:
        scratch = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
        off = (-scratch.data_ptr()) % 1024
        scratch = scratch[off:off + nbytes]
    check(load().wr_eval_rank_topk(ptr(Uemb, F32), ptr(Iemb, F32), ptr(user, I64), ptr(pos, I64), R,
                                   Uemb.shape[0], Iemb.shape[0], D, ptr(hist_ptr, I64), ptr(hist_idx, I32),
                                   k, precision, ptr(tki, I32), ptr(tkv, F32), ptr(rank, I32), ptr(target, F32),
                                   ptr(sc, F32), None if scratch is None else scratch.data_ptr(), ws.ptr,
                                   stream_ptr()))
    return rank, target, tki, tkv, sc


METRIC_CUTOFFS_PER_CALL = 8       # wr_metrics takes up to 8 cut-offs per launch
EVAL_DIMS = (16, 32, 64, 128, 256)     # embedding sizes the full-ranking evaluation kernels are instantiated for


def metrics(rank, ks, ws):
    """float64 tensor [2, len(ks)]: row 0 = HR@k, row 1 = NDCG@k (any number of cut-offs: 8 per launch)."""
    nk = len(ks)
    if nk <= METRIC_CUTOFFS_PER_CALL:
        out = torch.empty((2, nk), dtype=torch.float64, device=rank.device)
        arr = (ctypes.c_int * nk)(*[int(k) for k in ks])
        check(load().wr_metrics(ptr(rank, I32), rank.numel(), arr, nk, out.data_ptr(), ws.ptr, stream_ptr()))
        return out
    return torch.cat([metrics(rank, ks[c:c + METRIC_CUTOFFS_PER_CALL], ws) for c in range(0, nk, METRIC_CUTOFFS_PER_CALL)], dim=1)


def gather_rows(T, idx, ws, out=None):
    if out is None:
        out = torch.empty((idx.numel(), T.shape[1]), dtype=F32, device=T.device)
    check(load().wr_gather_rows(ptr(T, F32), ptr(idx, I64), idx.numel(), T.shape[1], T.shape[0], ptr(out, F32),
                                ws.ptr, stream_ptr()))
    return out


def scatter_add_rows(G, idx, rows, ws):
    check(load().wr_scatter_add_rows(ptr(G, F32), ptr(idx, I64), idx.numel(), G.shape[1], G.shape[0],
                                     ptr(rows, F32), ws.ptr, stream_ptr()))


def neg_sample_numpy_stream(user, n_users, n_items, train_ptr, train_idx, ws, scale=1):
    """One epoch of negatives on the device, consuming NumPy's GLOBAL legacy generator exactly as
    `np.random.randint` + the reference's redraw loop would (models/BaseModel.py:167-177); the global state is
    advanced accordingly.  user: int64 [N] device tensor; train_ptr / train_idx: device CSR.  Returns int64 [N]."""
    import numpy as np
    lib = load()
    N = user.numel()
    name, key, pos, has_gauss, cached = np.random.get_state()
    if name != 'MT19937':
        raise WhisprError('the global NumPy generator is not MT19937')
    key = np.ascontiguousarray(key, dtype=np.uint32)
    key_out = np.empty(624, dtype=np.uint32)
    pos_out = _int(0)
    neg = torch.empty(N, dtype=I64, device=user.device)
    nbytes = lib.wr_neg_sample_scratch_bytes(N, n_items) * scale
    scratch = torch.empty(nbytes + 16, dtype=torch.uint8, device=user.device)
    off = (-scratch.data_ptr()) % 16
    rc = lib.wr_neg_sample_mt19937(key.ctypes.data, int(pos), N, ptr(user, I64), n_users, n_items, ptr(train_ptr, I64),
                                   ptr(train_idx, I32), ptr(neg, I64), key_out.ctypes.data, ctypes.byref(pos_out),
                                   scratch.data_ptr() + off, nbytes, ws.ptr, stream_ptr())
    if rc == -2 and scale < 8:          # WR_E_SIZE: an unusually rejection-heavy draw; nothing was consumed yet
        return neg_sample_numpy_stream(user, n_users, n_items, train_ptr, train_idx, ws, scale * 2)
    check(rc)
    np.random.set_state((name, key_out, pos_out.value, has_gauss, cached))
    return neg


def py_random_sample(n, k):
    """`random.sample(range(n), k)` on Python's GLOBAL `random` generator, computed by the library (host code, same
    algorithm, same stream): returns an int64 NumPy array and leaves the generator where Python would."""
    import random
    import numpy as np
    version, internal, gauss = random.getstate()
    state = np.array(internal[:624], dtype=np.uint32)
    pos = _int(int(internal[624]))
    out = np.empty(int(k), dtype=np.int64)
    check(load().wr_pyrandom_sample(state.ctypes.data, ctypes.byref(pos), int(n), int(k), out.ctypes.data))
    random.setstate((version, tuple(int(x) for x in state) + (pos.value,), gauss))
    return out


# ------------------------------------------------------------------------------------------------------
# row-sharded tables over NVLink peer memory (include/whisprrec_b200.h, "one 8 x B200 box")
# ------------------------------------------------------------------------------------------------------
MAX_WORLD, PEER_VALUES = 8, 4


class ShardsStruct(ctypes.Structure):
    """Mirror of `wr_shards`."""
    _fields_ = [('base', _p * MAX_WORLD), ('world', _c.c_int32), ('rank', _c.c_int32), ('n_users', _i64),
                ('n_items', _i64), ('rows_u_local', _i64), ('rows_i_local', _i64)]


class PeerBlock:
    """A zero-filled cudaMalloc'd block that other processes on the box can map (cudaIpc*)."""

    def __init__(self, nbytes, device):
        self.device, self.nbytes = torch.device(device), int(nbytes)
        out = _p()
        with torch.cuda.device(self.device):
            check(load().wr_peer_alloc(self.nbytes, ctypes.byref(out)))
        self.ptr = out.value
        self._opened = []

    def handle(self):
        buf = ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            check(load().wr_peer_export(self.ptr, buf))
        return buf.raw

    def open_peer(self, handle):
        out = _p()
        with torch.cuda.device(self.device):
            check(load().wr_peer_open(handle, ctypes.byref(out)))
        self._opened.append(out.value)
        return out.value

    def tensor(self, offset, shape, dtype):
        """A torch view of [offset, offset + bytes) of the block (the block owns the memory)."""
        n = 1
        for d in shape:
            n *= int(d)
        itemsize = torch.empty((), dtype=dtype).element_size()
        assert offset % 16 == 0 and offset + n * itemsize <= self.nbytes
        typestr = {torch.float32: '<f4', torch.int32: '<i4', torch.uint32: '<u4', torch.int64: '<i8',
                   torch.uint8: '|u1'}[dtype]

        class _View:
            __cuda_array_interface__ = {'shape': tuple(int(d) for d in shape), 'typestr': typestr,
                                        'data': (self.ptr + offset, False), 'version': 2}
        v = _View()
        v._owner = self
        t = torch.as_tensor(v, device=self.device)
        t._wr_owner = self
        return t

    def close(self):
        lib = load()
        with torch.cuda.device(self.device):
            for p in self._opened:
                lib.wr_peer_close(p)
            self._opened = []
            if self.ptr:
                lib.wr_peer_free(self.ptr)
                self.ptr = None


def peer_barrier(flag_ptrs, slot_ptrs, world, rank, epoch, values_in=None, sums_out=None, ws=None):
    """flag_ptrs / slot_ptrs: lists of `world` raw device pointers (every rank's flag / slot array as mapped here)."""
    FA = _p * MAX_WORLD
    fa = FA(*(list(flag_ptrs) + [None] * (MAX_WORLD - world)))
    sa = FA(*(list(slot_ptrs) + [None] * (MAX_WORLD - world)))
    n = 0 if values_in is None else values_in.numel()
    check(load().wr_peer_barrier(ctypes.addressof(fa), world, rank, epoch, ctypes.addressof(sa), ptr(values_in, F32), n,
                                 ptr(sums_out, F32), None if ws is None else ws.ptr, stream_ptr()))


def bpr_fwd_bwd_sharded(T, Gd, user, pos, neg, B_global, D, loss_out, ws, gamma=1e-10, grad_scale=1.0):
    check(load().wr_bpr_fwd_bwd_sharded(ctypes.addressof(T), ctypes.addressof(Gd), ptr(user, I64), ptr(pos, I64),
                                        ptr(neg, I64), user.numel(), B_global, D, gamma, grad_scale,
                                        ptr(loss_out, F32), ws.ptr, stream_ptr()))


def bpr_fwd_bwd_sharded_staged(T, Gd, inbox_row_ptrs, inbox_idx_ptrs, cap, user, pos, neg, B_global, D, loss_out, ws,
                               gamma=1e-10, grad_scale=1.0):
    world = T.world
    FA = _p * MAX_WORLD
    ra = FA(*(list(inbox_row_ptrs) + [None] * (MAX_WORLD - world)))
    ia = FA(*(list(inbox_idx_ptrs) + [None] * (MAX_WORLD - world)))
    check(load().wr_bpr_fwd_bwd_sharded_staged(ctypes.addressof(T), ctypes.addressof(Gd), ctypes.addressof(ra),
                                               ctypes.addressof(ia), cap, ptr(user, I64), ptr(pos, I64), ptr(neg, I64),
                                               user.numel(), B_global, D, gamma, grad_scale, ptr(loss_out, F32), ws.ptr,
                                               stream_ptr()))


def _ptr_array(ptrs, world):
    FA = _p * MAX_WORLD
    return FA(*(list(ptrs) + [None] * (MAX_WORLD - world)))


def xchg_request(user, pos, neg, n_users, n_items, world, rank, req_ptrs, cnt_ptrs, cap, cnt_local, where, ws):
    ra, ca = _ptr_array(req_ptrs, world), _ptr_array(cnt_ptrs, world)
    check(load().wr_xchg_request(ptr(user, I64), ptr(pos, I64), ptr(neg, I64), user.numel(), n_users, n_items, world, rank,
                                 ctypes.addressof(ra), ctypes.addressof(ca), cap, ptr(cnt_local, I32), ptr(where, I32),
                                 ws.ptr, stream_ptr()))


def xchg_serve(T_local, world, rank, req_local, cnt_local, cap, recv_ptrs):
    va = _ptr_array(recv_ptrs, world)
    check(load().wr_xchg_serve(ptr(T_local, F32), T_local.shape[1], world, rank, ptr(req_local, I32), ptr(cnt_local, I32),
                               cap, ctypes.addressof(va), stream_ptr()))


def bpr_fwd_bwd_exchanged(recv, where, Gd, inbox_row_ptrs, inbox_idx_ptrs, cap, user, pos, neg, B_global, D, loss_out, ws,
                          gamma=1e-10, grad_scale=1.0, touched=None):
    world = Gd.world
    ra, ia = _ptr_array(inbox_row_ptrs, world), _ptr_array(inbox_idx_ptrs, world)
    check(load().wr_bpr_fwd_bwd_exchanged(ptr(recv, F32), ptr(where, I32), ctypes.addressof(Gd), ctypes.addressof(ra),
                                          ctypes.addressof(ia), cap, ptr(user, I64), ptr(pos, I64), ptr(neg, I64),
                                          user.numel(), B_global, D, gamma, grad_scale, ptr(touched, I32),
                                          ptr(loss_out, F32), ws.ptr, stream_ptr()))


def embloss_owner_sumsq(T_local, world, req_local, cnt_local, cap, sumsq_out, ws):
    check(load().wr_embloss_owner_sumsq(ptr(T_local, F32), T_local.shape[1], world, ptr(req_local, I32), ptr(cnt_local, I32),
                                        cap, ptr(sumsq_out, F32), ws.ptr, stream_ptr()))


def embloss_owner_scatter(T_local, G_local, world, req_local, cnt_local, cap, reg_weight, B_global, sumsq_global, loss_out):
    check(load().wr_embloss_owner_scatter(ptr(T_local, F32), ptr(G_local, F32), T_local.shape[1], world, ptr(req_local, I32),
                                          ptr(cnt_local, I32), cap, reg_weight, B_global, ptr(sumsq_global, F32),
                                          ptr(loss_out, F32), stream_ptr()))


def inbox_scatter(G, inbox_rows, inbox_idx, world, cap, touched=None):
    check(load().wr_inbox_scatter_marked(ptr(G, F32), ptr(inbox_rows, F32), ptr(inbox_idx, I32), world, cap, G.shape[1],
                                         ptr(touched, I32), stream_ptr()))


def push_marked_rows(X, D, node_bits, push_ptrs):
    """Store this rank's rows of the sharded table X whose GLOBAL node bit is set into every peer's copy of the shard."""
    pa = _ptr_array(push_ptrs, X.world)
    check(load().wr_push_marked_rows(ctypes.addressof(X), D, ptr(node_bits, I32), ctypes.addressof(pa), stream_ptr()))


def bprmf_step_sharded_supported(n_local_rows, D):
    return bool(load().wr_bprmf_step_sharded_supported(n_local_rows, D))


def bprmf_step_sharded(T, Gd, M, V, user, pos, neg, B_global, D, step, lr, l2, flag_ptrs, slot_ptrs, loss_out, ws,
                       beta1=0.9, beta2=0.999, eps=1e-8, gamma=1e-10, epoch=None):
    """One sharded BPRMF step in one cooperative launch.  `step` is Adam's t; `epoch` the synchronisation epoch
    (1, 2, 3, ... per table set; defaults to `step`)."""
    epoch = step if epoch is None else epoch
    world = T.world
    FA = _p * MAX_WORLD
    fa = FA(*(list(flag_ptrs) + [None] * (MAX_WORLD - world)))
    sa = FA(*(list(slot_ptrs) + [None] * (MAX_WORLD - world)))
    ss, bc2s = adam_scalars(step, lr, beta1, beta2)
    check(load().wr_bprmf_step_sharded(ctypes.addressof(T), ctypes.addressof(Gd), ptr(M, F32), ptr(V, F32),
                                       ptr(user, I64), ptr(pos, I64), ptr(neg, I64), user.numel(), B_global, D, gamma,
                                       l2, beta1, beta2, eps, ss, bc2s, epoch, ctypes.addressof(fa),
                                       ctypes.addressof(sa), ptr(loss_out, F32), ws.ptr, stream_ptr()))


def embloss_sumsq_sharded(T, user, pos, neg, D, sumsq_out, ws):
    check(load().wr_embloss_sumsq_sharded(ctypes.addressof(T), ptr(user, I64), ptr(pos, I64), ptr(neg, I64),
                                          user.numel(), D, ptr(sumsq_out, F32), ws.ptr, stream_ptr()))


def embloss_scatter_sharded(T, Gd, user, pos, neg, B_global, D, reg_weight, sumsq_global, loss_out, ws):
    check(load().wr_embloss_scatter_sharded(ctypes.addressof(T), ctypes.addressof(Gd), ptr(user, I64), ptr(pos, I64),
                                            ptr(neg, I64), user.numel(), B_global, D, reg_weight,
                                            ptr(sumsq_global, F32), ptr(loss_out, F32), ws.ptr, stream_ptr()))


def gather_rows_sharded(T, which, idx, D, ws, out=None):
    if out is None:
        out = torch.empty((idx.numel(), D), dtype=F32, device=idx.device)
    check(load().wr_gather_rows_sharded(ctypes.addressof(T), which, ptr(idx, I64), idx.numel(), D, ptr(out, F32),
                                        ws.ptr, stream_ptr()))
    return out


def allgather_shards(src, dst, D):
    check(load().wr_allgather_shards(ctypes.addressof(src), ptr(dst, F32), D, stream_ptr()))


def csr_spmm_sharded(rowptr, col, val, n_local, D, X, Y=None, add=None, zero_add=False, acc_in=None, acc_out=None,
                     acc_div=1.0, plan=None, push_ptrs=None, x_rows=None):
    """push_ptrs: list of `world` raw pointers (entry [rank] ignored / None): every peer's copy of this rank's shard of Y,
    written from the SpMM epilogue (the fused all-gather).  x_rows: bitmap over the GLOBAL node ids (the column ids)."""
    pa = None
    keep = []
    if push_ptrs is not None:
        FA = _p * MAX_WORLD
        pa = FA(*(list(push_ptrs) + [None] * (MAX_WORLD - len(push_ptrs))))
    check(load().wr_csr_spmm_sharded(ptr(rowptr, I64), ptr(col, I32), ptr(val, F32), n_local, D, ctypes.addressof(X),
                                     ptr(Y, F32), ptr(add, F32), int(zero_add), ptr(acc_in, F32), ptr(acc_out, F32),
                                     acc_div, _plan_ref(plan, x_rows, keep),
                                     None if pa is None else ctypes.addressof(pa), stream_ptr()))


def csr_spmm_sharded_dma(rowptr, col, val, n_local, D, X, Y, push_ptrs, progress, block_rows, epoch, side_stream, nnz=0,
                         add=None, zero_add=False, acc_in=None, acc_out=None, acc_div=1.0, plan=None, x_rows=None):
    """csr_spmm_sharded with the all-gather of Y done by the copy engines on `side_stream` while the kernel runs."""
    pa = _ptr_array(push_ptrs, X.world)
    keep = []
    check(load().wr_csr_spmm_sharded_dma(ptr(rowptr, I64), ptr(col, I32), ptr(val, F32), n_local, D, ctypes.addressof(X),
                                         ptr(Y, F32), ptr(add, F32), int(zero_add), ptr(acc_in, F32), ptr(acc_out, F32),
                                         acc_div, _plan_ref(plan, x_rows, keep), ctypes.addressof(pa), ptr(progress, I32),
                                         progress.numel(), block_rows, epoch, nnz, side_stream.cuda_stream, stream_ptr()))


def push_shard_dma(src, world, rank, push_ptrs):
    pa = _ptr_array(push_ptrs, world)
    check(load().wr_push_shard_dma(ptr(src, F32), src.numel(), world, rank, ctypes.addressof(pa), stream_ptr()))


def rowdot(A, B, round_bf16=False):
    out = torch.empty(A.shape[0], dtype=F32, device=A.device)
    check(load().wr_rowdot(ptr(A, F32), ptr(B, F32), A.shape[0], A.shape[1], int(round_bf16), ptr(out, F32),
                           stream_ptr()))
    return out


def eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k=0, precision=0):
    """One item shard: returns (rank int32 [R] = 1 + local count, topk_idx LOCAL int32 [R,k] | None, topk_val | None).
    Precision 2 with k, and k up to 256, as in eval_rank_topk."""
    R, D = user.numel(), Urows.shape[1]
    if k > TOPK_KMAX:
        return _eval_rank_topk_long_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k,
                                          _long_precision(D, k, precision, False))
    if precision == 2 and k > 0:
        if not exact_tc_topk_supported(D, k):
            return _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k, 0)
        out = _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k, 2)
        st = ws.status()
        ws.last_topk_fallback_rows = 0
        if st & 4:
            out = _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k, 0)
            ws.last_topk_fallback_rows = R
        elif st & 8:
            _exact_topk_fallback(out[1:3], Urows, True, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k)
        st &= ~12
        if st:
            ws.restore_status(st)
        return out
    if precision == 2:
        if not exact_tc_supported(D, k):
            precision = 0
        else:
            out = _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, 0, 2)
            st = ws.status()
            if st & 4:
                out = _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, 0, 0)
                st &= ~4
            if st:
                ws.restore_status(st)
            return out
    return _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k, precision)


def _eval_rank_topk_shard(Urows, Iemb, user, pos_local, n_users, hist_ptr, hist_idx, target, ws, k, precision):
    R, D = user.numel(), Urows.shape[1]
    dev = Urows.device
    rank = torch.empty(R, dtype=I32, device=dev)
    tki = torch.empty((R, k), dtype=I32, device=dev) if k > 0 else None
    tkv = torch.empty((R, k), dtype=F32, device=dev) if k > 0 else None
    nbytes = load().wr_eval_scratch_bytes_topk(R, Iemb.shape[0], D, precision, k)
    scratch = None
    if nbytes:
        scratch = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
        off = (-scratch.data_ptr()) % 1024
        scratch = scratch[off:off + nbytes]
    check(load().wr_eval_rank_topk_shard(ptr(Urows, F32), ptr(Iemb, F32), ptr(user, I64), ptr(pos_local, I64), R,
                                         n_users, Iemb.shape[0], D, ptr(hist_ptr, I64), ptr(hist_idx, I32), k,
                                         precision, ptr(target, F32), ptr(tki, I32), ptr(tkv, F32), ptr(rank, I32),
                                         None if scratch is None else scratch.data_ptr(), ws.ptr, stream_ptr()))
    return rank, tki, tkv


def topk_merge(val, idx, k):
    """val / idx: [world, R, k] candidates with GLOBAL item ids -> ([R, k] values, [R, k] ids); k up to 256."""
    world, R = val.shape[0], val.shape[1]
    ov = torch.empty((R, k), dtype=F32, device=val.device)
    oi = torch.empty((R, k), dtype=I32, device=val.device)
    merge = load().wr_topk_merge_long if k > TOPK_KMAX else load().wr_topk_merge
    check(merge(ptr(val, F32), ptr(idx, I32), world, R, k, ptr(ov, F32), ptr(oi, I32), stream_ptr()))
    return ov, oi
