"""Row-sharded kernels on one GPU: `world` emulated ranks against the single-GPU kernels.

A kernel of the sharded path only loads, stores and reduces through the `wr_shards` base pointers; it cannot tell a
peer mapping from an ordinary allocation on its own device.  So the tests below allocate every rank's shards on one
device, build one `wr_shards` per emulated rank and issue the ranks' calls in protocol order on one stream: stream order
stands in for the cross-GPU barriers.  What this checks is the owner arithmetic -- owners, local rows, padding rows,
request lists, receive slots, inbox slots, row maps -- at worlds 1 to 8, not the memory model of real peer memory.

The two kernels that wait on other ranks (wr_peer_barrier and the single-launch sharded step) and the copy-engine SpMM
push (a stream wait on a flag the kernel sets) are never reached here: the module replaces them with functions that
raise.  They stay with the multi-GPU tests.

CPU: argument errors of the sharded entry points on fake pointers (nothing is launched).
GPU: every entry point against the single-GPU kernel or a float64 reference; the drivers of sharded.py (the body of
`tests/dist_worker.py gpu`) with ranks in threads.
"""
import random
import threading

import numpy as np
import pytest
import torch

from tests.helpers import assert_close
from whisprrec_b200 import _lib
from whisprrec_b200 import sharded as S

WR_E_NULL, WR_E_SIZE, WR_E_DIM, WR_E_ALIGN = -1, -2, -3, -5
OUT_OF_RANGE = 1                       # WR_STATUS_INDEX_OUT_OF_RANGE
WORLDS = (1, 2, 3, 8)                  # 8 = WR_MAX_WORLD; 3 pads unevenly
FAST_DIMS = (16, 32, 64, 128, 256)
RED_TOL = dict(rtol=1e-5, atol_scale=2e-6)     # sums whose order depends on the REDs' arrival order
SENTINEL = -7.25


# ---------------------------------------------------------------------------------------------------------
# CPU: argument errors on fake pointers
# ---------------------------------------------------------------------------------------------------------

def fake_shards(n_users=10, n_items=7, world=2, rank=0, rows_u_local=None, rows_i_local=None, base=None):
    s = _lib.ShardsStruct()
    for g in range(min(world, _lib.MAX_WORLD)):
        s.base[g] = 4096 * (g + 1) if base is None else base[g]
    s.world, s.rank, s.n_users, s.n_items = world, rank, n_users, n_items
    s.rows_u_local = -(-n_users // world) if rows_u_local is None else rows_u_local
    s.rows_i_local = -(-n_items // world) if rows_i_local is None else rows_i_local
    return s


def ptrs(*p):
    """A wr_* pointer array of WR_MAX_WORLD entries."""
    return _lib._ptr_array(p, len(p))


def addr(x):
    import ctypes
    return ctypes.addressof(x)


F = 1 << 16                            # a fake, 16-byte aligned device address


def test_sharded_table_argument_errors():
    lib = _lib.load()
    good = fake_shards()
    bad_u = fake_shards(rows_u_local=4)                 # ceil(10 / 2) = 5
    bad_i = fake_shards(rows_i_local=3)                 # ceil(7 / 2) = 4
    # wr_bpr_fwd_bwd_sharded(T, Gd, user, pos, neg, B, B_global, D, gamma, grad_scale, loss, ws, stream)
    bpr = lambda T, Gd, B=4, Bg=8, D=64: lib.wr_bpr_fwd_bwd_sharded(addr(T), addr(Gd), F, F, F, B, Bg, D, 1e-10, 1.0,
                                                                     F, F, None)
    assert bpr(bad_u, good) == WR_E_SIZE and bpr(good, bad_u) == WR_E_SIZE and bpr(good, bad_i) == WR_E_SIZE
    assert bpr(good, good, B=5, Bg=4) == WR_E_SIZE and bpr(good, good, B=0) == WR_E_SIZE
    assert bpr(good, good, D=18) == WR_E_DIM and bpr(good, good, D=0) == WR_E_DIM
    assert bpr(fake_shards(world=9), good) == WR_E_SIZE
    assert bpr(fake_shards(rank=2), good) == WR_E_SIZE
    assert bpr(fake_shards(n_users=0, rows_u_local=0), good) == WR_E_SIZE
    assert bpr(fake_shards(base=[F, 0]), good) == WR_E_NULL
    assert bpr(fake_shards(base=[F, F + 4]), good) == WR_E_ALIGN
    assert lib.wr_bpr_fwd_bwd_sharded(addr(good), addr(good), None, F, F, 4, 8, 64, 1e-10, 1.0, F, F, None) == WR_E_NULL

    rows, idx = ptrs(F, F), ptrs(F, F)
    # wr_bpr_fwd_bwd_sharded_staged(T, Gd, inbox_rows, inbox_idx, cap, user, pos, neg, B, B_global, D, gamma,
    #                               grad_scale, loss, ws, stream)
    staged = lambda D=64, cap=12, B=4, r=rows, T=good: lib.wr_bpr_fwd_bwd_sharded_staged(
        addr(T), addr(good), addr(r), addr(idx), cap, F, F, F, B, 8, D, 1e-10, 1.0, F, F, None)
    assert staged(D=48) == WR_E_DIM and staged(D=20) == WR_E_DIM and staged(D=512) == WR_E_DIM
    assert staged(cap=11) == WR_E_SIZE and staged(T=bad_u) == WR_E_SIZE
    assert staged(r=ptrs(F, F + 8)) == WR_E_ALIGN and staged(r=ptrs(F, 0)) == WR_E_NULL
    # wr_bpr_fwd_bwd_exchanged(recv, where, Gd, inbox_rows, inbox_idx, cap, user, pos, neg, B, B_global, D, gamma,
    #                          grad_scale, touched, loss, ws, stream)
    xchg = lambda D=64, cap=12, recv=F, Gd=good, Bg=8: lib.wr_bpr_fwd_bwd_exchanged(
        recv, F, addr(Gd), addr(rows), addr(idx), cap, F, F, F, 4, Bg, D, 1e-10, 1.0, None, F, F, None)
    assert xchg(D=48) == WR_E_DIM and xchg(cap=11) == WR_E_SIZE and xchg(Bg=3) == WR_E_SIZE
    assert xchg(recv=F + 4) == WR_E_ALIGN and xchg(recv=None) == WR_E_NULL and xchg(Gd=bad_i) == WR_E_SIZE

    # wr_embloss_sumsq_sharded(T, user, pos, neg, B, D, sumsq, ws, stream)
    assert lib.wr_embloss_sumsq_sharded(addr(bad_u), F, F, F, 4, 64, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_sumsq_sharded(addr(good), F, F, F, 0, 64, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_sumsq_sharded(addr(good), F, F, F, 4, 18, F, F, None) == WR_E_DIM
    # wr_embloss_scatter_sharded(T, Gd, user, pos, neg, B, B_global, D, reg, sumsq_global, loss, ws, stream)
    assert lib.wr_embloss_scatter_sharded(addr(good), addr(bad_i), F, F, F, 4, 8, 64, 1e-5, F, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_scatter_sharded(addr(good), addr(good), F, F, F, 4, 3, 64, 1e-5, F, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_scatter_sharded(addr(good), addr(good), F, F, F, 4, 8, 64, 1e-5, None, F, F, None) == WR_E_NULL

    # wr_gather_rows_sharded(T, which, idx, B, D, out, ws, stream): B = 0 is a no-op (nothing is launched)
    assert lib.wr_gather_rows_sharded(addr(good), 2, F, 4, 64, F, F, None) == WR_E_SIZE
    assert lib.wr_gather_rows_sharded(addr(good), 0, F, 4, 18, F, F, None) == WR_E_DIM
    assert lib.wr_gather_rows_sharded(addr(good), 1, F, 4, 64, F + 4, F, None) == WR_E_ALIGN
    assert lib.wr_gather_rows_sharded(addr(bad_u), 0, F, 4, 64, F, F, None) == WR_E_SIZE
    assert lib.wr_gather_rows_sharded(addr(good), 0, F, 0, 64, F, F, None) == 0
    # wr_allgather_shards(src, dst, D, stream): world 1 has nothing to gather
    assert lib.wr_allgather_shards(addr(good), F + 4, 64, None) == WR_E_ALIGN
    assert lib.wr_allgather_shards(addr(good), F, 18, None) == WR_E_DIM
    assert lib.wr_allgather_shards(addr(bad_i), F, 64, None) == WR_E_SIZE
    assert lib.wr_allgather_shards(addr(fake_shards(world=1)), F, 64, None) == 0


def test_exchange_argument_errors():
    lib = _lib.load()
    req, cnt = ptrs(F, F, F), ptrs(F, F, F)
    # wr_xchg_request(user, pos, neg, B, n_users, n_items, world, rank, req, cnt, cap, cnt_local, where, ws, stream)
    rq = lambda B=4, world=3, rank=0, cap=12, r=req: lib.wr_xchg_request(F, F, F, B, 10, 7, world, rank, addr(r),
                                                                           addr(cnt), cap, F, F, F, None)
    assert rq(cap=11) == WR_E_SIZE and rq(B=0) == WR_E_SIZE and rq(world=9) == WR_E_SIZE and rq(rank=3) == WR_E_SIZE
    assert rq(world=0) == WR_E_SIZE and rq(r=ptrs(F, None, F)) == WR_E_NULL
    assert lib.wr_xchg_request(F, F, F, 4, 10, 7, 3, 0, addr(req), addr(cnt), 12, None, F, F, None) == WR_E_NULL
    # wr_xchg_serve(T, D, world, rank, req, cnt, cap, recv, stream)
    sv = lambda D=64, world=3, rank=0, cap=12, recv=ptrs(F, F, F): lib.wr_xchg_serve(F, D, world, rank, F, F, cap,
                                                                                     addr(recv), None)
    assert sv(D=18) == WR_E_DIM and sv(cap=0) == WR_E_SIZE and sv(rank=-1) == WR_E_SIZE and sv(world=9) == WR_E_SIZE
    assert sv(recv=ptrs(F, F + 8, F)) == WR_E_ALIGN and sv(recv=ptrs(F, None, F)) == WR_E_NULL
    # wr_embloss_owner_sumsq(T, D, world, req, cnt, cap, sumsq, ws, stream)
    assert lib.wr_embloss_owner_sumsq(F, 18, 3, F, F, 12, F, F, None) == WR_E_DIM
    assert lib.wr_embloss_owner_sumsq(F, 64, 0, F, F, 12, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_owner_sumsq(F, 64, 3, F, F, 0, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_owner_sumsq(F, 64, 3, F, F, 12, None, F, None) == WR_E_NULL
    # wr_embloss_owner_scatter(T, G, D, world, req, cnt, cap, reg, B_global, sumsq_global, loss, stream)
    assert lib.wr_embloss_owner_scatter(F, F, 64, 3, F, F, 12, 1e-5, 0, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_owner_scatter(F, F, 20 + 2, 3, F, F, 12, 1e-5, 8, F, F, None) == WR_E_DIM
    assert lib.wr_embloss_owner_scatter(F, F + 4, 64, 3, F, F, 12, 1e-5, 8, F, F, None) == WR_E_ALIGN
    # wr_inbox_scatter(_marked)(G, rows, idx, world, cap, D, [touched,] stream)
    assert lib.wr_inbox_scatter(F, F, F, 9, 12, 64, None) == WR_E_SIZE
    assert lib.wr_inbox_scatter(F, F, F, 3, 0, 64, None) == WR_E_SIZE
    assert lib.wr_inbox_scatter(F, F, F, 3, 12, 18, None) == WR_E_DIM
    assert lib.wr_inbox_scatter_marked(F, F + 4, F, 3, 12, 64, F, None) == WR_E_ALIGN
    assert lib.wr_inbox_scatter_marked(None, F, F, 3, 12, 64, F, None) == WR_E_NULL
    # wr_push_marked_rows(X, D, node_bits, push, stream): no peer to push to is a no-op
    good = fake_shards(world=3)
    assert lib.wr_push_marked_rows(addr(good), 18, F, addr(ptrs(None, F, F)), None) == WR_E_DIM
    assert lib.wr_push_marked_rows(addr(good), 64, F, addr(ptrs(None, F, F + 4)), None) == WR_E_ALIGN
    assert lib.wr_push_marked_rows(addr(fake_shards(world=3, rows_u_local=3)), 64, F, addr(ptrs(None, F, F)),
                                   None) == WR_E_SIZE
    assert lib.wr_push_marked_rows(addr(good), 64, F, addr(ptrs(F, None, None)), None) == 0
    assert lib.wr_push_marked_rows(addr(fake_shards(world=1)), 64, F, addr(ptrs(F)), None) == 0
    # wr_mark_rows(user, pos, neg, B, n_users, n_items, touched, stream)
    assert lib.wr_mark_rows(F, F, F, 0, 10, 7, F, None) == WR_E_SIZE
    assert lib.wr_mark_rows(F, F, None, 4, 10, 7, F, None) == WR_E_NULL
    with pytest.raises(_lib.WhisprError, match='row map too small'):
        _lib.mark_rows(None, None, None, 10, 7, torch.zeros(0, dtype=torch.int32))


def test_spmm_push_rowdot_embloss_argument_errors():
    lib = _lib.load()
    good = fake_shards(world=2)                       # n_local = 5 + 4
    # wr_csr_spmm_sharded(rowptr, col, val, n_local, D, X, Y, add, zero_add, acc_in, acc_out, acc_div, plan, push, stream)
    sp = lambda n_local=9, D=64, X=good, Y=F, acc_out=None, push=None: lib.wr_csr_spmm_sharded(
        F, F, F, n_local, D, addr(X), Y, None, 0, F, acc_out, 1.0, None, None if push is None else addr(push), None)
    assert sp(n_local=8) == WR_E_SIZE and sp(n_local=10) == WR_E_SIZE
    assert sp(D=18) == WR_E_DIM and sp(X=fake_shards(world=2, rows_i_local=5)) == WR_E_SIZE
    assert sp(Y=4096) == WR_E_SIZE                         # Y is the rank's own shard of X
    assert sp(Y=None) == WR_E_NULL                         # nothing to write
    assert sp(Y=None, acc_out=F, push=ptrs(None, F)) == WR_E_NULL     # a push needs Y
    assert sp(push=ptrs(None, F + 4)) == WR_E_ALIGN and sp(Y=F + 4) == WR_E_ALIGN
    # wr_push_shard_dma(src, n_floats, world, rank, push, stream): world 1 copies nothing
    assert lib.wr_push_shard_dma(F, 64, 9, 0, addr(ptrs(F)), None) == WR_E_SIZE
    assert lib.wr_push_shard_dma(F, 0, 2, 0, addr(ptrs(None, F)), None) == WR_E_SIZE
    assert lib.wr_push_shard_dma(F, 64, 2, 2, addr(ptrs(None, F)), None) == WR_E_SIZE
    assert lib.wr_push_shard_dma(None, 64, 2, 0, addr(ptrs(None, F)), None) == WR_E_NULL
    assert lib.wr_push_shard_dma(F, 64, 1, 0, addr(ptrs(F)), None) == 0
    # wr_rowdot(A, B, R, D, round_bf16, out, stream)
    assert lib.wr_rowdot(F, F, 0, 64, 0, F, None) == WR_E_SIZE and lib.wr_rowdot(F, F, -1, 64, 1, F, None) == WR_E_SIZE
    assert lib.wr_rowdot(F, F, 4, 18, 0, F, None) == WR_E_DIM and lib.wr_rowdot(F, F, 4, 0, 1, F, None) == WR_E_DIM
    assert lib.wr_rowdot(F + 4, F, 4, 64, 0, F, None) == WR_E_ALIGN and lib.wr_rowdot(F, F, 4, 64, 0, None, None) == WR_E_NULL
    # wr_embloss_fwd_bwd(U0, I0, user, pos, neg, B, D, n_users, n_items, reg, gU0, gI0, loss, ws, stream)
    assert lib.wr_embloss_fwd_bwd(F, F, F, F, F, 0, 64, 10, 7, 1e-5, F, F, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_fwd_bwd(F, F, F, F, F, 4, 64, 0, 7, 1e-5, F, F, F, F, None) == WR_E_SIZE
    assert lib.wr_embloss_fwd_bwd(F, F, F, F, F, 4, 18, 10, 7, 1e-5, F, F, F, F, None) == WR_E_DIM
    assert lib.wr_embloss_fwd_bwd(F, F, F, F, F, 4, 64, 10, 7, 1e-5, F, F + 4, F, F, None) == WR_E_ALIGN
    assert lib.wr_embloss_fwd_bwd(F, F, F, F, F, 4, 64, 10, 7, 1e-5, F, F, None, F, None) == WR_E_NULL


# ---------------------------------------------------------------------------------------------------------
# GPU: emulated ranks
# ---------------------------------------------------------------------------------------------------------

DEV = torch.device('cuda:0')


@pytest.fixture(autouse=True)
def no_spinning_paths(monkeypatch):
    """Ranks that wait on each other must never share a GPU: the paths that spin are unreachable in this module."""
    def refuse(*a, **k):
        raise AssertionError('a cross-rank wait was reached with emulated ranks on one GPU')
    monkeypatch.setattr(_lib, 'peer_barrier', refuse)
    monkeypatch.setattr(_lib, 'bprmf_step_sharded', refuse)
    monkeypatch.setattr(_lib, 'csr_spmm_sharded_dma', refuse)
    monkeypatch.setattr(_lib, 'bprmf_step_sharded_supported', lambda *a: False)
    monkeypatch.setenv('WR_SPMM_PUSH', 'store')


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def host(t):
    return t.detach().cpu().numpy()


class Emulated(object):
    """`world` ranks of one sharded layout on one device: layouts, one workspace per rank, and helpers that cut a full
    [n_users + n_items, D] table into its shards and describe them with one wr_shards per rank."""

    def __init__(self, n_users, n_items, world):
        self.n_users, self.n_items, self.world = n_users, n_items, world
        self.lay = [S.ShardLayout(n_users, n_items, world, r) for r in range(world)]
        self.n_local = self.lay[0].n_local
        self.ws = [_lib.Workspace(DEV) for _ in range(world)]
        self._keep = []                   # tensors behind the wr_shards built here live as long as this object


    def shards(self, full):
        return [lay.shard_of_table(full) for lay in self.lay]

    def zeros(self, D):
        return [torch.zeros((self.n_local, D), dtype=torch.float32, device=DEV) for _ in range(self.world)]

    def structs(self, tensors):
        self._keep.append(tensors)
        out = []
        for r, lay in enumerate(self.lay):
            s = _lib.ShardsStruct()
            for g, t in enumerate(tensors):
                s.base[g] = t.data_ptr()
            s.world, s.rank, s.n_users, s.n_items = self.world, r, self.n_users, self.n_items
            s.rows_u_local, s.rows_i_local = lay.rows_u_local, lay.rows_i_local
            out.append(s)
        return out

    def full_of(self, shards):
        """The full table behind a list of shards (host arithmetic: inverse of shard_of_table)."""
        D = shards[0].shape[1]
        full = torch.zeros((self.n_users + self.n_items, D), dtype=torch.float32, device=DEV)
        for lay, t in zip(self.lay, shards):
            nodes = lay.local_nodes()
            ok = np.nonzero(nodes >= 0)[0]
            full[torch.from_numpy(nodes[ok]).to(DEV)] = t[torch.from_numpy(ok).to(DEV)]
        return full

    def padding(self, t, r):
        return t[torch.from_numpy(np.nonzero(self.lay[r].local_nodes() < 0)[0]).to(DEV)]

    def statuses(self):
        return [ws.status() for ws in self.ws]


def tables(n_users, n_items, D, seed, zero_items=()):
    """Distinct rows; users, positives (first half of the items) and negatives (second half) on different scales, so
    that a swapped role or owner changes the numbers."""
    rng = np.random.RandomState(seed)
    U = rng.randn(n_users, D) * 0.5 + np.arange(n_users)[:, None] * 1e-3
    I = rng.randn(n_items, D) * 0.05 + np.arange(n_items)[:, None] * 1e-4
    I[n_items // 2:] *= 4.0
    I[list(zero_items)] = 0.0
    return U.astype(np.float32), I.astype(np.float32)


def batch(n_users, n_items, B, seed, bad=False, neg_from=None):
    """Positives from the first half of the items, negatives from the second; duplicate ids; with bad=True one entry
    has an out-of-range negative."""
    rng = np.random.RandomState(seed + 1)
    half = max(1, n_items // 2)
    user = rng.randint(0, n_users, B)
    pos = rng.randint(0, half, B)
    neg = rng.randint(half, n_items, B) if neg_from is None else rng.choice(neg_from, B)
    # duplicates in every role; at most ~B/50 copies of one row, so that fp32 sums of a row's contributions stay within
    # 1e-5 of the float64 reference (n equal addends round to ~n/2 ulp)
    user[B // 2:B // 2 + 3] = user[0]
    pos[1::61], neg[2::53] = pos[0], neg[0]
    if bad:
        neg[B // 3] = n_items
    return user.astype(np.int64), pos.astype(np.int64), neg.astype(np.int64)


def valid_entries(user, pos, neg, n_users, n_items):
    return (user >= 0) & (user < n_users) & (pos >= 0) & (pos < n_items) & (neg >= 0) & (neg < n_items)


# Shapes: n_users < world at worlds 3 and 8 (ranks whose only user row is padding); n_items % world != 0;
# B % world != 0.
SHAPES = ((2, 203, 1001), (301, 517, 2050))


def check_slices_status(em, B, bad_at):
    """The out-of-range bit is raised by exactly the rank whose slice holds the bad entry."""
    st = em.statuses()
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        assert st[r] == (OUT_OF_RANGE if bad_at is not None and lo <= bad_at < hi else 0), (r, st)


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
def test_gather_rows_and_allgather(world):
    for nU, nI, _ in SHAPES:
        D = 20 if nU < 10 else 64
        U, I = tables(nU, nI, D, 1)
        full = dev(np.concatenate([U, I]))
        em = Emulated(nU, nI, world)
        sh = em.shards(full)
        T = em.structs(sh)
        for r in range(world):
            for which, n, want in ((0, nU, full[:nU]), (1, nI, full[nU:])):
                idx = torch.cat([torch.arange(n, device=DEV), torch.tensor([n - 1, 0, n], device=DEV)])
                got = _lib.gather_rows_sharded(T[r], which, idx, D, em.ws[r])
                assert torch.equal(got[:n], want) and torch.equal(got[n:n + 2], want[[n - 1, 0]])
                assert float(got[n + 2].abs().max()) == 0.0
                assert em.ws[r].status() == OUT_OF_RANGE
        for r in range(world):
            dst = torch.full((world, em.n_local, D), SENTINEL, device=DEV)
            _lib.allgather_shards(T[r], dst, D)
            for g in range(world):
                assert torch.equal(dst[g], sh[g]) if g != r else bool((dst[g] == SENTINEL).all()), (r, g)
        assert em.statuses() == [0] * world


def bpr_reference(U, I, user, pos, neg, D, ws):
    gU, gI = torch.zeros_like(U), torch.zeros_like(I)
    loss = torch.zeros(1, device=DEV)
    _lib.bpr_fwd_bwd(U, I, user, pos, neg, gU, gI, loss, ws)
    return float(loss[0]), gU, gI


def check_gradient(em, G, gU, gI, what):
    full = em.full_of(G)
    Gd = em.structs(G)[0]
    D = gU.shape[1]
    gu = _lib.gather_rows_sharded(Gd, 0, torch.arange(em.n_users, device=DEV), D, em.ws[0])
    gi = _lib.gather_rows_sharded(Gd, 1, torch.arange(em.n_items, device=DEV), D, em.ws[0])
    assert torch.equal(gu, full[:em.n_users]) and torch.equal(gi, full[em.n_users:])
    assert_close(host(gu), host(gU), what + ' user gradient', **RED_TOL)
    assert_close(host(gi), host(gI), what + ' item gradient', **RED_TOL)
    for r in range(em.world):
        pad = em.padding(G[r], r)
        assert pad.numel() == 0 or float(pad.abs().max()) == 0.0, 'gradient in a padding row'


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
@pytest.mark.parametrize('D', FAST_DIMS + (20, 48))
def test_bpr_fwd_bwd_sharded(world, D):
    for si, (nU, nI, B) in enumerate(SHAPES):
        U, I = tables(nU, nI, D, 2 + si)
        user, pos, neg = batch(nU, nI, B, 3 + si, bad=True)
        Ud, Id = dev(U), dev(I)
        ud, pd, nd = dev(user), dev(pos), dev(neg)
        ref_ws = _lib.Workspace(DEV)
        loss, gU, gI = bpr_reference(Ud, Id, ud, pd, nd, D, ref_ws)
        assert ref_ws.status() == OUT_OF_RANGE
        em = Emulated(nU, nI, world)
        T = em.structs(em.shards(torch.cat([Ud, Id])))
        G = em.zeros(D)
        Gd = em.structs(G)
        parts = []
        for r, lay in enumerate(em.lay):
            lo, hi = lay.batch_slice(B)
            lp = torch.zeros(_lib.PEER_VALUES, device=DEV)
            _lib.bpr_fwd_bwd_sharded(T[r], Gd[r], ud[lo:hi], pd[lo:hi], nd[lo:hi], B, D, lp[:1], em.ws[r])
            parts.append(float(lp[0]))
        check_slices_status(em, B, B // 3)
        assert abs(sum(parts) - loss) <= 2e-6 * abs(loss), (sum(parts), loss)
        check_gradient(em, G, gU, gI, f'sharded world {world} D {D}')


def inbox(em, D, cap):
    rows = [torch.zeros((em.world, cap, D), device=DEV) for _ in range(em.world)]
    idx = [torch.zeros((em.world, cap), dtype=torch.int32, device=DEV) for _ in range(em.world)]
    return rows, idx, [t.data_ptr() for t in rows], [t.data_ptr() for t in idx]


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
@pytest.mark.parametrize('D', FAST_DIMS)
def test_bpr_fwd_bwd_sharded_staged(world, D):
    nU, nI, B = SHAPES[1]
    U, I = tables(nU, nI, D, 4)
    user, pos, neg = batch(nU, nI, B, 5, bad=True)
    Ud, Id, ud, pd, nd = dev(U), dev(I), dev(user), dev(pos), dev(neg)
    loss, gU, gI = bpr_reference(Ud, Id, ud, pd, nd, D, _lib.Workspace(DEV))
    em = Emulated(nU, nI, world)
    T = em.structs(em.shards(torch.cat([Ud, Id])))
    G = em.zeros(D)
    Gd = em.structs(G)
    cap = 3 * -(-B // world)
    rows, idx, row_ptrs, idx_ptrs = inbox(em, D, cap)
    total = 0.0
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        lp = torch.zeros(1, device=DEV)
        _lib.bpr_fwd_bwd_sharded_staged(T[r], Gd[r], row_ptrs, idx_ptrs, cap, ud[lo:hi], pd[lo:hi], nd[lo:hi], B, D, lp,
                                        em.ws[r])
        total += float(lp[0])
    check_slices_status(em, B, B // 3)
    for o in range(world):
        _lib.inbox_scatter(G[o], rows[o], idx[o], world, cap)
        assert int(idx[o].abs().max()) == 0
    assert abs(total - loss) <= 2e-6 * abs(loss), (total, loss)
    check_gradient(em, G, gU, gI, f'staged world {world} D {D}')
    if D == 64:
        lp = torch.zeros(1, device=DEV)
        with pytest.raises(_lib.WhisprError, match='error -3'):
            _lib.bpr_fwd_bwd_sharded_staged(T[0], Gd[0], row_ptrs, idx_ptrs, cap, ud[:4], pd[:4], nd[:4], B, 48, lp,
                                            em.ws[0])


class Exchange(object):
    """The symmetric buffers of the row exchange for every emulated rank (what ShardedTables.exchange allocates)."""

    def __init__(self, em, D, B):
        w = em.world
        self.cap = cap = 3 * -(-B // w)
        self.req = [torch.zeros((w, cap), dtype=torch.int32, device=DEV) for _ in range(w)]
        self.cnt = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(w)]
        self.recv = [torch.full((w, cap, D), SENTINEL, device=DEV) for _ in range(w)]
        self.cnt_local = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(w)]
        self.where = [torch.zeros(cap, dtype=torch.int32, device=DEV) for _ in range(w)]
        self.req_ptrs = [t.data_ptr() for t in self.req]
        self.cnt_ptrs = [t.data_ptr() for t in self.cnt]
        self.recv_ptrs = [t.data_ptr() for t in self.recv]

    def request(self, em, ud, pd, nd, B):
        for r, lay in enumerate(em.lay):
            lo, hi = lay.batch_slice(B)
            _lib.xchg_request(ud[lo:hi], pd[lo:hi], nd[lo:hi], em.n_users, em.n_items, em.world, r, self.req_ptrs,
                              self.cnt_ptrs, self.cap, self.cnt_local[r], self.where[r], em.ws[r])
        for r in range(em.world):
            assert int(self.cnt_local[r].abs().max()) == 0          # ready for the next step

    def serve(self, em, shards):
        for o in range(em.world):
            _lib.xchg_serve(shards[o], em.world, o, self.req[o], self.cnt[o], self.cap, self.recv_ptrs)


def request_model(em, user, pos, neg, B):
    """NumPy model of the request lists: want[o][r] = sorted (local_row << 2 | role) that requester r sends owner o."""
    w, ok = em.world, valid_entries(user, pos, neg, em.n_users, em.n_items)
    want = [[[] for _ in range(w)] for _ in range(w)]
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        for b in range(lo, hi):
            if not ok[b]:
                continue
            for role, (i, off) in enumerate(((user[b], 0), (pos[b], lay.rows_u_local), (neg[b], lay.rows_u_local))):
                want[i % w][r].append(((off + i // w) << 2) | role)
    return [[np.sort(np.array(x, dtype=np.int64)) for x in row] for row in want]


def check_requests(em, x, user, pos, neg, B):
    want = request_model(em, user, pos, neg, B)
    for o in range(em.world):
        cnt = host(x.cnt[o])
        for r in range(em.world):
            got = np.sort(host(x.req[o][r, :cnt[r]]).astype(np.int64))
            assert np.array_equal(got, want[o][r]), (o, r)


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
@pytest.mark.parametrize('D', FAST_DIMS)
def test_exchange_step(world, D):
    """request -> serve -> exchanged fwd/bwd with the row map -> inbox scatter -> row-marked Adam, rank by rank."""
    nU, nI, B = SHAPES[1] if D != 16 else SHAPES[0]
    U, I = tables(nU, nI, D, 6)
    user, pos, neg = batch(nU, nI, B, 7, bad=True)
    Ud, Id, ud, pd, nd = dev(U), dev(I), dev(user), dev(pos), dev(neg)
    loss, gU, gI = bpr_reference(Ud, Id, ud, pd, nd, D, _lib.Workspace(DEV))
    em = Emulated(nU, nI, world)
    full = torch.cat([Ud, Id])
    P = em.shards(full)
    x = Exchange(em, D, B)
    x.request(em, ud, pd, nd, B)
    check_slices_status(em, B, B // 3)
    check_requests(em, x, user, pos, neg, B)
    x.serve(em, P)
    ok = valid_entries(user, pos, neg, nU, nI)
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        where = host(x.where[r])
        recv = x.recv[r].reshape(-1, D)
        for role, ids, base in ((0, user, 0), (1, pos, nU), (2, neg, nU)):
            bs = np.nonzero(ok[lo:hi])[0]
            got = recv[dev(where[3 * bs + role].astype(np.int64))]
            assert torch.equal(got, full[dev(base + ids[lo + bs])]), (r, role)
    G = em.zeros(D)
    Gd = em.structs(G)
    rows, idx, row_ptrs, idx_ptrs = inbox(em, D, x.cap)
    touched = [_lib.row_map(em.n_local, DEV) for _ in range(world)]
    total = 0.0
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        lp = torch.zeros(1, device=DEV)
        _lib.bpr_fwd_bwd_exchanged(x.recv[r], x.where[r], Gd[r], row_ptrs, idx_ptrs, x.cap, ud[lo:hi], pd[lo:hi],
                                   nd[lo:hi], B, D, lp, em.ws[r], touched=touched[r])
        total += float(lp[0])
    check_slices_status(em, B, B // 3)
    for o in range(world):
        _lib.inbox_scatter(G[o], rows[o], idx[o], world, x.cap, touched[o])
        assert int(idx[o].abs().max()) == 0
    assert abs(total - loss) <= 2e-6 * abs(loss), (total, loss)
    check_gradient(em, G, gU, gI, f'exchanged world {world} D {D}')
    # the row maps: exactly the local rows that received a gradient (entries with every id in range)
    nodes_hit = np.zeros(nU + nI, dtype=bool)
    nodes_hit[user[ok]] = True
    nodes_hit[nU + pos[ok]] = True
    nodes_hit[nU + neg[ok]] = True
    rng = np.random.RandomState(8)
    for o, lay in enumerate(em.lay):
        nodes = lay.local_nodes()
        want = np.where(nodes >= 0, nodes_hit[np.maximum(nodes, 0)], False)
        bits = np.unpackbits(host(touched[o]).view(np.uint8), bitorder='little')[:em.n_local].astype(bool)
        assert np.array_equal(bits, want), o
        assert not np.unpackbits(host(touched[o]).view(np.uint8), bitorder='little')[em.n_local:].any()
        # the row-marked sweep on the shard equals the dense sweep on the same G, bit for bit
        M = dev((rng.randn(em.n_local, D) * 1e-3).astype(np.float32))
        V = dev((rng.rand(em.n_local, D) * 1e-4).astype(np.float32))
        dense = [t.clone() for t in (P[o], M, V, G[o])]
        _lib.adam_l2_sweep(*dense, 3, 1e-3, 1e-4)
        _lib.adam_l2_sweep_marked(P[o], M, V, G[o], touched[o], 3, 1e-3, 1e-4)
        for a, b in zip((P[o], M, V, G[o]), dense):
            assert torch.equal(a, b), o
        assert int(touched[o].abs().max()) == 0
    with pytest.raises(_lib.WhisprError, match='error -3'):
        _lib.bpr_fwd_bwd_exchanged(x.recv[0], x.where[0], Gd[0], row_ptrs, idx_ptrs, x.cap, ud[:4], pd[:4], nd[:4], B,
                                   48, torch.zeros(1, device=DEV), em.ws[0])


def embloss_reference(U, I, user, pos, neg, reg):
    """EmbLoss (utils/loss.py:83-98) in float64 over the entries with every id in range; B counts every entry."""
    U, I = U.astype(np.float64), I.astype(np.float64)
    B = len(user)
    ok = valid_entries(user, pos, neg, len(U), len(I))
    gU, gI = np.zeros_like(U), np.zeros_like(I)
    loss = 0.0
    for ids, tab, g in ((user, U, gU), (pos, I, gI), (neg, I, gI)):
        X = tab[ids[ok]]
        n = np.sqrt((X * X).sum())
        loss += n
        if n > 0:
            np.add.at(g, ids[ok], reg / B * X / n)
    return reg * loss / B, gU, gI


EMB_CASES = ('duplicates', 'zero_negatives', 'out_of_range')


def emb_case(nU, nI, D, B, case, seed):
    zero = list(range(nI - 5, nI)) if case == 'zero_negatives' else []
    U, I = tables(nU, nI, D, seed, zero_items=zero)
    user, pos, neg = batch(nU, nI, B, seed, bad=case == 'out_of_range' and B > 1, neg_from=zero or None)
    if case == 'out_of_range' and B == 1:
        user[0] = nU
    return U, I, user, pos, neg


@pytest.mark.gpu
@pytest.mark.parametrize('case', EMB_CASES)
@pytest.mark.parametrize('D', (16, 64, 256, 20))
@pytest.mark.parametrize('B', (1, 33, 4096))
def test_embloss_fwd_bwd(B, D, case):
    nU, nI, reg = 97, 211, 1e-3
    U, I, user, pos, neg = emb_case(nU, nI, D, B, case, 11)
    ws = _lib.Workspace(DEV)
    gU, gI = torch.zeros((nU, D), device=DEV), torch.zeros((nI, D), device=DEV)
    loss = torch.zeros(1, device=DEV)
    _lib.embloss_fwd_bwd(dev(U), dev(I), dev(user), dev(pos), dev(neg), gU, gI, loss, ws, reg)
    assert ws.status() == 0            # skipped, not reported: the BPR kernel of the same step reports it
    want_loss, want_gU, want_gI = embloss_reference(U, I, user, pos, neg, reg)
    assert np.isfinite(host(gU)).all() and np.isfinite(host(gI)).all()
    assert abs(float(loss[0]) - want_loss) <= 1e-5 * abs(want_loss) + 1e-30, (float(loss[0]), want_loss)
    assert_close(host(gU), want_gU, 'EmbLoss user gradient', **RED_TOL)
    assert_close(host(gI), want_gI, 'EmbLoss item gradient', **RED_TOL)
    if case == 'zero_negatives':
        assert float(gI[nI - 5:].abs().max()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
@pytest.mark.parametrize('case', EMB_CASES)
@pytest.mark.parametrize('D', (16, 64, 256))
def test_embloss_sharded_and_owner(world, case, D):
    """Remote form (sums of squares per rank's slice, scatter by REDs) and owner form (from the request lists)."""
    nU, nI, B, reg = 5, 203, 1001, 1e-3
    U, I, user, pos, neg = emb_case(nU, nI, D, B, case, 13)
    ud, pd, nd = dev(user), dev(pos), dev(neg)
    want_loss, want_gU, want_gI = embloss_reference(U, I, user, pos, neg, reg)
    em = Emulated(nU, nI, world)
    P = em.shards(dev(np.concatenate([U, I])))
    T = em.structs(P)
    bad_at = B // 3 if case == 'out_of_range' else None

    # remote form: every rank reads its slice's rows from their owners
    G = em.zeros(D)
    Gd = em.structs(G)
    part = [torch.zeros(_lib.PEER_VALUES, device=DEV) for _ in range(world)]
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        _lib.embloss_sumsq_sharded(T[r], ud[lo:hi], pd[lo:hi], nd[lo:hi], D, part[r][:3], em.ws[r])
    sums = torch.zeros(_lib.PEER_VALUES, device=DEV)
    for p in part:                      # what wr_peer_barrier returns: the ranks' values added in rank order
        sums = sums + p
    for r, lay in enumerate(em.lay):
        lo, hi = lay.batch_slice(B)
        lr = torch.zeros(1, device=DEV)
        _lib.embloss_scatter_sharded(T[r], Gd[r], ud[lo:hi], pd[lo:hi], nd[lo:hi], B, D, reg, sums, lr, em.ws[r])
        assert abs(float(lr[0]) - want_loss) <= 1e-5 * abs(want_loss) + 1e-30, (r, float(lr[0]), want_loss)
    check_slices_status(em, B, None)    # as embloss_fwd_bwd: skipped, not reported
    check_gradient(em, G, torch.from_numpy(want_gU.astype(np.float32)).to(DEV),
                   torch.from_numpy(want_gI.astype(np.float32)).to(DEV), f'EmbLoss sharded world {world}')

    # owner form: the owners of the ego rows compute from the request lists of the exchange
    x = Exchange(em, D, B)
    x.request(em, ud, pd, nd, B)
    check_slices_status(em, B, bad_at)
    G = em.zeros(D)
    part = [torch.zeros(_lib.PEER_VALUES, device=DEV) for _ in range(world)]
    for o in range(world):
        _lib.embloss_owner_sumsq(P[o], world, x.req[o], x.cnt[o], x.cap, part[o][:3], em.ws[o])
    sums = torch.zeros(_lib.PEER_VALUES, device=DEV)
    for p in part:
        sums = sums + p
    for o in range(world):
        lo_ = torch.zeros(1, device=DEV)
        _lib.embloss_owner_scatter(P[o], G[o], world, x.req[o], x.cnt[o], x.cap, reg, B, sums, lo_)
        assert abs(float(lo_[0]) - want_loss) <= 1e-5 * abs(want_loss) + 1e-30, (o, float(lo_[0]), want_loss)
    check_gradient(em, G, torch.from_numpy(want_gU.astype(np.float32)).to(DEV),
                   torch.from_numpy(want_gI.astype(np.float32)).to(DEV), f'EmbLoss owners world {world}')
    assert em.statuses() == [0] * world


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
def test_mark_rows_and_push_marked_rows(world):
    nU, nI, B, D = 301, 517, 700, 64
    U, I = tables(nU, nI, D, 15)
    user, pos, neg = batch(nU, nI, B, 16, bad=True)
    N = nU + nI
    gm = _lib.row_map(N, DEV)
    _lib.mark_rows(dev(user), dev(pos), dev(neg), nU, nI, gm)
    ok = valid_entries(user, pos, neg, nU, nI)
    want = np.zeros(N, dtype=bool)
    want[user[ok]] = want[nU + pos[ok]] = want[nU + neg[ok]] = True
    bits = np.unpackbits(host(gm).view(np.uint8), bitorder='little').astype(bool)
    assert np.array_equal(bits[:N], want) and not bits[N:].any()
    em = Emulated(nU, nI, world)
    P = em.shards(dev(np.concatenate([U, I])))
    T = em.structs(P)
    for r, lay in enumerate(em.lay):
        copies = [torch.full((em.n_local, D), SENTINEL, device=DEV) for _ in range(world)]
        _lib.push_marked_rows(T[r], D, gm, [None if g == r else copies[g].data_ptr() for g in range(world)])
        nodes = lay.local_nodes()
        marked = dev(np.where(nodes >= 0, want[np.maximum(nodes, 0)], False))
        for g in range(world):
            if g == r:
                assert bool((copies[g] == SENTINEL).all())
                continue
            assert torch.equal(copies[g][marked], P[r][marked])
            assert bool((copies[g][~marked] == SENTINEL).all())


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
def test_push_shard_dma(world):
    D = 32
    em = Emulated(301, 517, world)
    P = em.shards(dev(np.concatenate(tables(301, 517, D, 17))))
    for r in range(world):
        copies = [torch.full((em.n_local, D), SENTINEL, device=DEV) for _ in range(world)]
        _lib.push_shard_dma(P[r], world, r, [None if g == r else copies[g].data_ptr() for g in range(world)])
        for g in range(world):
            assert torch.equal(copies[g], P[r]) if g != r else bool((copies[g] == SENTINEL).all())


def power_law_graph(nU, nI, seed):
    """Bipartite interactions where a few users and items have far more than 128 neighbours (split SpMM rows)."""
    rng = np.random.RandomState(seed)
    u = np.concatenate([rng.randint(0, nU, 3000), np.zeros(700, np.int64), np.full(300, 3), rng.randint(0, nU, 400)])
    i = np.concatenate([rng.zipf(1.6, 3000) % nI, rng.randint(0, nI, 700), rng.randint(0, nI, 300),
                        np.full(400, 7)])
    return u.astype(np.int64), i.astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
@pytest.mark.parametrize('D', (16, 64, 128, 256, 20))
def test_csr_spmm_sharded(world, D):
    from oracle import whispr_oracle as O
    nU, nI = 450, 1413
    N = nU + nI
    u, i = power_law_graph(nU, nI, 19)
    rowptr, col, val = O.build_norm_adj_csr(nU, nI, u, i)
    deg = np.diff(rowptr)
    assert deg[:nU].max() > 3 * 128 and deg[nU:].max() > 128        # split user rows and split item rows
    rng = np.random.RandomState(21)
    X = dev(rng.randn(N, D).astype(np.float32))
    add = dev(rng.randn(N, D).astype(np.float32))
    acc_in = dev(rng.randn(N, D).astype(np.float32))
    marked = rng.rand(N) < 0.3
    x_rows = dev(np.packbits(np.pad(marked, (0, (-N) % 32)), bitorder='little').view(np.int32))
    rp, cl, vl = dev(rowptr), dev(col.astype(np.int32)), dev(val.astype(np.float32))
    # single-GPU references (no plan: no row is split)
    Y1 = torch.zeros_like(X)
    add1 = add.clone()
    _lib.csr_spmm(rp, cl, vl, X, Y=Y1, add=add1, zero_add=True)
    acc1 = torch.zeros_like(X)
    _lib.csr_spmm(rp, cl, vl, X, acc_in=acc_in, acc_out=acc1, acc_div=3.0, x_rows=x_rows)

    em = Emulated(nU, nI, world)
    Xs = em.structs(em.shards(X))
    split_possible = D in FAST_DIMS
    for r, lay in enumerate(em.lay):
        lptr, lcol, src = lay.local_adjacency(rowptr, col)
        nodes = lay.local_nodes()
        okr = nodes >= 0
        lrp, lcl = dev(lptr), dev(lcol if len(lcol) else np.zeros(1, np.int32))
        lvl = dev(val[src].astype(np.float32) if len(src) else np.zeros(1, np.float32))
        plan = _lib.SpmmPlan(lptr, D, DEV)
        split = (np.diff(lptr) > plan.threshold) & split_possible
        assert plan.n_long == int((np.diff(lptr) > plan.threshold).sum())
        exact, tol = dev(okr & ~split), dev(okr & split)
        pad = dev(~okr)
        want_rows = dev(np.maximum(nodes, 0))

        def compare(got, ref, what):
            assert torch.equal(got[exact], ref[want_rows][exact]), what
            if bool(tol.any()):
                assert_close(host(got[tol]), host(ref[want_rows][tol]), what, **RED_TOL)

        Y = torch.zeros((em.n_local, D), device=DEV)
        add_r = lay.shard_of_table(add)
        copies = [torch.full((em.n_local, D), SENTINEL, device=DEV) for _ in range(world)]
        push = [None if g == r else copies[g].data_ptr() for g in range(world)]
        _lib.csr_spmm_sharded(lrp, lcl, lvl, em.n_local, D, Xs[r], Y=Y, add=add_r, zero_add=True, plan=plan,
                              push_ptrs=push)
        compare(Y, Y1, f'Y + add, rank {r}')
        assert not bool(pad.any()) or float(Y[pad].abs().max()) == 0.0
        assert float(add_r.abs().max()) == 0.0                          # zero_add clears the addend
        for g in range(world):
            assert torch.equal(copies[g], Y) if g != r else bool((copies[g] == SENTINEL).all())

        acc_r = torch.zeros((em.n_local, D), device=DEV)
        _lib.csr_spmm_sharded(lrp, lcl, lvl, em.n_local, D, Xs[r], acc_in=lay.shard_of_table(acc_in), acc_out=acc_r,
                              acc_div=3.0, plan=plan, x_rows=x_rows)
        compare(acc_r, acc1, f'layer mean with x_rows, rank {r}')


def full_scores_target_case(D, seed):
    rng = np.random.RandomState(seed)
    nU, nI, R = 61, 700, 257
    U = (rng.randn(nU, D) * 0.3).astype(np.float32)
    I = (rng.randn(nI, D) * 0.3).astype(np.float32)
    user, pos = rng.randint(0, nU, R).astype(np.int64), rng.randint(0, nI, R).astype(np.int64)
    hist_ptr, hist_idx = np.zeros(nU + 1, dtype=np.int64), np.zeros(1, dtype=np.int32)
    return dev(U), dev(I), dev(user), dev(pos), dev(hist_ptr), dev(hist_idx)


@pytest.mark.gpu
@pytest.mark.parametrize('precision,D', [(0, d) for d in FAST_DIMS] + [(2, d) for d in (64, 128, 256)] +
                         [(1, d) for d in (64, 128, 256)])
def test_rowdot_reproduces_the_eval_target(precision, D):
    """sharded_eval scores the target with rowdot: it has to be the single-GPU kernels' target bit for bit, or the ranks
    of near-ties differ."""
    U, I, user, pos, hp, hi = full_scores_target_case(D, 23 + D)
    ws = _lib.Workspace(DEV)
    want = _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, precision=precision)[1]
    assert ws.status() == 0
    got = _lib.rowdot(U[user].contiguous(), I[pos].contiguous(), round_bf16=precision == 1)
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------------
# GPU: the drivers of sharded.py, one thread per emulated rank
# ---------------------------------------------------------------------------------------------------------

class _Meeting(object):
    """What the emulated ranks share.  Between two collective calls exactly one rank runs (in rank order), with its own
    state of the host generators (NumPy's, torch's, Python's) swapped in: every rank draws as a process of its own
    would.  At a collective call a rank finishes its device work, posts its contribution, hands the turn on and meets
    the others at a threading.Barrier."""

    def __init__(self, world, timeout, device_sync=True):
        self.world, self.timeout, self.device_sync = world, timeout, device_sync
        self.barrier = threading.Barrier(world, timeout=timeout)
        self.cond = threading.Condition()
        self.turn, self.failed = 0, False
        self.posts = [[None] * world, [None] * world]
        self.rng = [self._rng_state()] * world

    @staticmethod
    def _rng_state():
        return np.random.get_state(), torch.get_rng_state(), random.getstate()

    def wait_turn(self, rank):
        with self.cond:
            if not self.cond.wait_for(lambda: self.failed or self.turn == rank, self.timeout):
                raise TimeoutError('rank %d never got its turn' % rank)
            if self.failed:
                raise threading.BrokenBarrierError
            np_state, torch_state, py_state = self.rng[rank]
            np.random.set_state(np_state)
            torch.set_rng_state(torch_state)
            random.setstate(py_state)

    def pass_turn(self, rank):
        with self.cond:
            self.rng[rank] = self._rng_state()
            self.turn = (rank + 1) % self.world
            self.cond.notify_all()

    def fail(self):
        with self.cond:
            self.failed = True
            self.cond.notify_all()
        self.barrier.abort()

    def collective(self, rank, n, value):
        """The n-th collective call of `rank`: every rank's value, in rank order."""
        if self.device_sync:
            torch.cuda.synchronize()
        slot = self.posts[n & 1]            # a rank is at most one call ahead of the slowest reader
        slot[rank] = value
        self.pass_turn(rank)
        self.barrier.wait()
        self.wait_turn(rank)
        return list(slot)


class _HostPeers(object):
    """A rank of the meeting with no device: rank, world and the host rendezvous."""

    def __init__(self, meeting, rank):
        self.meeting, self.rank, self.world = meeting, rank, meeting.world
        self._n = 0

    def _collective(self, value):
        self._n += 1
        return self.meeting.collective(self.rank, self._n, value)

    def host_sync(self):
        self._collective(None)


class _FakeDist(object):
    """The torch.distributed calls of sharded.py, within the emulated ranks."""

    def __init__(self, group):
        self.g = group

    def all_reduce(self, t, group=None):
        total = None
        for v in self.g._collective(t.clone()):
            total = v if total is None else total + v
        t.copy_(total)

    def all_gather_into_tensor(self, out, t, group=None):
        out.copy_(torch.stack(self.g._collective(t.clone())).reshape(out.shape))

    def barrier(self, group=None):
        self.g._collective(None)


class FakePeerGroup(_HostPeers):
    """PeerGroup's interface for one emulated rank: symmetric allocations are ordinary allocations on the one device,
    and the device-side barrier is a host meeting after a device synchronisation (what stream order on one GPU needs)."""

    def __init__(self, meeting, rank):
        super().__init__(meeting, rank)
        torch.cuda.set_device(DEV)                  # the current device is per thread
        self.device = DEV
        self.group = None
        self.dist = _FakeDist(self)
        self.ws = _lib.Workspace(DEV)
        self.sums = torch.zeros(_lib.PEER_VALUES, dtype=torch.float32, device=DEV)
        self._keep = []

    def alloc_bytes(self, nbytes):
        t = torch.zeros(int(nbytes), dtype=torch.uint8, device=DEV)
        self._keep.append(t)
        return t, self._collective(t.data_ptr())

    def alloc(self, shape, dtype=torch.float32):
        t = torch.zeros(tuple(int(d) for d in shape), dtype=dtype, device=DEV)
        self._keep.append(t)
        return t, self._collective(t.data_ptr())

    def barrier(self, values=None):
        posted = self._collective(None if values is None else values.clone())
        if values is None:
            return None
        n = values.numel()
        total = torch.zeros(n, dtype=torch.float32, device=DEV)
        for v in posted:                     # peer_barrier_kernel: t = 0; t += value of rank r, r = 0 .. world-1
            total = total + v
        self.sums[:n].copy_(total)
        return self.sums[:n]

    def close(self):
        self.host_sync()
        self.ws.raise_on_status()


def run_ranks(world, body, make_peers=FakePeerGroup, device_sync=True, timeout=900.0):
    """body(peers) on `world` threads, one make_peers(meeting, rank) each.  A failing rank aborts the meeting, so the
    others end too; every thread is joined before this returns, and the first error that is not the abort is raised."""
    meeting = _Meeting(world, timeout, device_sync)
    errors = [None] * world

    def main(rank):
        try:
            meeting.wait_turn(rank)
            body(make_peers(meeting, rank))
            meeting.pass_turn(rank)
        except BaseException as e:  # noqa: BLE001 - re-raised on the test's thread
            errors[rank] = e
            meeting.fail()
    threads = [threading.Thread(target=main, args=(r,), name='emulated-rank-%d' % r) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout)
    if any(t.is_alive() for t in threads):
        meeting.fail()
        for t in threads:
            t.join(60.0)
    assert not any(t.is_alive() for t in threads), 'emulated ranks did not finish'
    real = [e for e in errors if e is not None and not isinstance(e, threading.BrokenBarrierError)]
    if real:
        raise real[0]
    assert not any(errors), errors


@pytest.mark.gpu
@pytest.mark.parametrize('world', [2, 3])
def test_sharded_drivers_with_emulated_ranks(world, capsys):
    """The per-rank body of `torchrun ... tests/dist_worker.py gpu` (bprmf_step on both multi-launch protocols,
    ShardedLightGCN.step with pull all-gather, copy-engine push, store push, exchange and sparse pooled gradient,
    sharded_eval at k = 10 and 100, model.shard with an ml-100k epoch against the goldens) on emulated ranks."""
    from tests.dist_worker import check_sharded_paths

    def body(peers):
        check_sharded_paths(peers)
        peers.close()
    run_ranks(world, body)
    out = capsys.readouterr().out
    assert out.count('dist_worker gpu ok') == 5, out


def test_emulated_ranks_take_turns_and_end_on_a_failing_rank():
    """Between meetings one rank runs at a time, in rank order, with generators of its own; a rank that raises ends
    every rank (no hang, no thread left behind) and its error is the one reported."""
    order, draws = [], [[] for _ in range(3)]

    def body(peers):
        np.random.seed(5)
        for step in range(3):
            order.append((step, peers.rank))
            draws[peers.rank].append(np.random.randint(1 << 30))
            peers.host_sync()
    run_ranks(3, body, make_peers=_HostPeers, device_sync=False, timeout=30.0)
    assert order == [(s, r) for s in range(3) for r in range(3)]
    assert draws[0] == draws[1] == draws[2] and len(set(draws[0])) == 3      # every rank its own generator

    def failing(peers):
        peers.host_sync()
        if peers.rank == 1:
            raise ValueError('rank 1 fails')
        peers.host_sync()
    before = threading.active_count()
    with pytest.raises(ValueError, match='rank 1 fails'):
        run_ranks(3, failing, make_peers=_HostPeers, device_sync=False, timeout=30.0)
    assert threading.active_count() == before
