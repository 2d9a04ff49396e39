"""SGL on row shards: the sharded InfoNCE (wr_infonce_sharded_*), the sum-form BPR on shards, and whole SGL steps and
epochs through `model.shard()` -- emulated ranks on one GPU (tests/test_sharded_emulated.py) against the single-GPU path.

CPU: argument errors of the new entry points on fake pointers (nothing is launched); the per-rank row cuts of an
edge-dropout view and of its transpose tile the whole view.
"""
import random

import numpy as np
import pytest
import torch

from tests.helpers import assert_close, frames_corpus, load, ml100k_corpus, model_args, small_case
from tests.test_sharded_emulated import (DEV, F, RED_TOL, WORLDS, WR_E_ALIGN, WR_E_DIM, WR_E_NULL, WR_E_SIZE, Emulated,
                                         addr, batch, dev, fake_shards, host, no_spinning_paths, ptrs, run_ranks, tables)
from whisprrec_b200 import _lib
from whisprrec_b200 import sharded as S

assert no_spinning_paths          # the autouse fixture of the emulated-rank module applies here too


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------

def test_sharded_sgl_argument_errors():
    lib = _lib.load()
    good = fake_shards(world=2)
    z, ga = ptrs(F, F), ptrs(F, F)
    # wr_infonce_sharded_partials(T1, T2, which, idx, B, D, tau, z, scratch, scratch_bytes, ws, stream)
    part = lambda T1=good, T2=good, which=0, idx=F, B=4, D=64, tau=0.1, zz=z, nbytes=1 << 30: \
        lib.wr_infonce_sharded_partials(addr(T1), addr(T2), which, idx, B, D, tau, addr(zz), F, nbytes, F, None)
    assert part(D=18) == WR_E_DIM and part(D=260) == WR_E_DIM and part(D=0) == WR_E_DIM
    assert part(B=0) == WR_E_SIZE and part(tau=0.0) == WR_E_SIZE and part(which=2) == WR_E_SIZE
    assert part(T2=fake_shards(world=2, rows_u_local=4)) == WR_E_SIZE
    assert part(T1=fake_shards(world=2, rank=1)) == WR_E_SIZE            # T1 and T2 describe different ranks
    assert part(T1=fake_shards(world=9)) == WR_E_SIZE
    assert part(T2=fake_shards(world=2, base=[F, 0])) == WR_E_NULL
    assert part(zz=ptrs(F, None)) == WR_E_NULL and part(idx=None) == WR_E_NULL
    assert part(nbytes=lib.wr_infonce_sharded_scratch_bytes(4, 5, 64) - 1) == WR_E_SIZE
    # wr_infonce_sharded_weights(dT2, which, idx, B, D, tau, weight, grad_scale, z, ga, loss, scratch, bytes, stream)
    wts = lambda dT2=good, D=64, B=4, gg=ga, loss=F: lib.wr_infonce_sharded_weights(
        addr(dT2), 1, F, B, D, 0.1, 0.05, 1.0, addr(z), addr(gg), loss, F, 1 << 30, None)
    assert wts(D=20 + 2) == WR_E_DIM and wts(B=-1) == WR_E_SIZE and wts(dT2=fake_shards(world=2, rows_i_local=5)) == WR_E_SIZE
    assert wts(gg=ptrs(F, F + 4)) == WR_E_ALIGN and wts(gg=ptrs(None, F)) == WR_E_NULL and wts(loss=None) == WR_E_NULL
    # wr_infonce_sharded_batch(dT1, which, idx, B, D, tau, weight, grad_scale, ga, scratch, bytes, stream)
    bat = lambda D=64, gg=ga, nbytes=1 << 30: lib.wr_infonce_sharded_batch(addr(good), 0, F, 4, D, 0.1, 0.05, 1.0, addr(gg),
                                                                          F, nbytes, None)
    assert bat(D=512) == WR_E_DIM and bat(gg=ptrs(F + 8, F)) == WR_E_ALIGN and bat(nbytes=16) == WR_E_SIZE
    # the scratch query: 0 for what the calls refuse; grows with the local rows, not with B x N
    q = lib.wr_infonce_sharded_scratch_bytes
    assert q(0, 5, 64) == 0 and q(4, -1, 64) == 0 and q(4, 5, 18) == 0 and q(4, 5, 260) == 0
    assert q(4, 0, 64) > 0                                               # a rank with no rows of the block
    assert q(2048, 10 ** 6, 64) < 2 * 10 ** 6 * 64 * 4 + 64 * 2048 * 64 * 4
    # wr_bpr_logsig_sum_fwd_bwd_sharded(T, Gd, user, pos, neg, B, B_global, D, grad_scale, loss, ws, stream)
    bpr = lambda T=good, B=4, Bg=8, D=64, loss=F: lib.wr_bpr_logsig_sum_fwd_bwd_sharded(addr(T), addr(good), F, F, F, B,
                                                                                       Bg, D, 1.0, loss, F, None)
    assert bpr(B=5, Bg=4) == WR_E_SIZE and bpr(B=0) == WR_E_SIZE and bpr(D=18) == WR_E_DIM
    assert bpr(T=fake_shards(world=2, rows_u_local=4)) == WR_E_SIZE and bpr(loss=None) == WR_E_NULL


def view_case(nU, nI, seed, drop=0.1):
    """A random bipartite train set, its normalised adjacency and one host edge-dropout view (and transpose)."""
    from whisprrec_b200.models.general.LightGCN import build_norm_adj_csr
    from whisprrec_b200.utils import graph_views
    rng = np.random.RandomState(seed)
    pairs = np.unique(np.stack([rng.randint(0, nU, 6 * (nU + nI)), rng.randint(0, nI, 6 * (nU + nI))], 1), axis=0)
    ptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(np.bincount(pairs[:, 0], minlength=nU), out=ptr[1:])
    rowptr, col, _ = build_norm_adj_csr(nU, nI, ptr, pairs[:, 1].astype(np.int32))
    random.seed(seed)
    return graph_views.edge_dropout_view(rowptr, col, drop, transpose=True)


def host_cut(lay, g):
    """A rank's rows of a global host CSR (rowptr, col, val), as LocalGraph cuts them on the device."""
    lptr, lcol, src = lay.local_adjacency(g[0], g[1])
    return lptr, lcol, np.asarray(g[2])[src]


@pytest.mark.parametrize('world', WORLDS)
def test_view_row_cuts_tile_the_view(world):
    """sharded.local_rows -- the cut LocalGraph runs on the device, here on CPU tensors -- gives every row of a view and
    of its transpose to exactly one rank, bit for bit, in local row order (and agrees with ShardLayout.local_adjacency)."""
    for nU, nI, seed in ((2, 40, 3), (57, 31, 4)):            # n_users < world at world 3 / 8
        fwd, tr = view_case(nU, nI, seed)
        for g in (fwd, tr):
            rowptr = np.asarray(g[0])
            seen = np.zeros(nU + nI, dtype=int)
            for r in range(world):
                lay = S.ShardLayout(nU, nI, world, r)
                lptr_t, lcol_t, src, _, _ = S.local_rows(lay, torch.from_numpy(rowptr), torch.from_numpy(np.asarray(g[1])))
                lptr, lcol, lval = lptr_t.numpy(), lcol_t.numpy(), np.asarray(g[2])[src.numpy()]
                hptr, hcol, hval = host_cut(lay, g)
                assert (lptr == hptr).all() and (lcol == hcol).all() and lval.tobytes() == hval.tobytes()
                assert len(lptr) == lay.n_local + 1
                for l, node in enumerate(lay.local_nodes()):
                    a, b = lptr[l], lptr[l + 1]
                    if node < 0:
                        assert a == b
                        continue
                    seen[node] += 1
                    lo, hi = rowptr[node], rowptr[node + 1]
                    assert (lcol[a:b] == g[1][lo:hi]).all()
                    assert lval[a:b].tobytes() == np.asarray(g[2][lo:hi]).tobytes()
            assert (seen == 1).all()


# ---------------------------------------------------------------------------------------------------------
# GPU: the sharded InfoNCE against wr_infonce_fwd_bwd
# ---------------------------------------------------------------------------------------------------------

def infonce_sharded(em, T1, T2, which, idx, D, tau, w, gs):
    """The three phases on every emulated rank, in protocol order.  Returns (per-rank losses, full dT1, full dT2)."""
    B, world = idx.numel(), em.world
    S1, S2 = em.structs(em.shards(T1)), em.structs(em.shards(T2))
    d1, d2 = em.zeros(D), em.zeros(D)
    G1, G2 = em.structs(d1), em.structs(d2)
    z = [torch.full((world, B), float('nan'), device=DEV) for _ in range(world)]
    ga = [torch.full((world, B, D), float('nan'), device=DEV) for _ in range(world)]
    zp, gp = [t.data_ptr() for t in z], [t.data_ptr() for t in ga]
    loss = [torch.zeros(1, device=DEV) for _ in range(world)]
    sc = [_lib.infonce_sharded_scratch(B, len(lay.local_users() if which == 0 else lay.local_items()), D, DEV)
          for lay in em.lay]
    for r in range(world):
        _lib.infonce_sharded_partials(S1[r], S2[r], which, idx, D, tau, zp, sc[r], em.ws[r])
    for r in range(world):
        _lib.infonce_sharded_weights(G2[r], which, idx, D, tau, w, gs, zp, gp, loss[r], sc[r])
    for r in range(world):
        _lib.infonce_sharded_batch(G1[r], which, idx, D, tau, w, gs, gp, sc[r])
    for r in range(world):
        for t in (d1[r], d2[r]):
            pad = em.padding(t, r)
            assert pad.numel() == 0 or float(pad.abs().max()) == 0.0, 'gradient in a padding row'
    return [float(l[0]) for l in loss], em.full_of(d1), em.full_of(d2)


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
@pytest.mark.parametrize('D', [16, 20, 64, 256])
def test_infonce_sharded_matches_single_gpu(world, D):
    # 2 users: ranks with no user rows at worlds 3 and 8 (that shape stops at B = 65: thousands of copies of one id
    # would sum beyond the RED tolerance in any order)
    for si, (nU, nI, Bs) in enumerate(((2, 203, (1, 65)), (301, 517, (1, 65, 2048)))):
        U, I = tables(nU, nI, D, 7 + si)
        T1 = dev(np.concatenate([U, I]))
        T2 = dev(np.concatenate(tables(nU, nI, D, 17 + si)))     # independent views: no dominant positive pair
        for B in Bs:
            user, pos, _ = batch(nU, nI, B, 5 + si + B) if B > 3 else (np.arange(B) % nU, np.arange(B) % nI, None)
            for tau in (0.1, 0.5):
                for which, ids, rows in ((0, user, slice(0, nU)), (1, pos, slice(nU, nU + nI))):
                    idx = dev(ids)
                    ref_loss = torch.zeros(1, device=DEV)
                    r1, r2 = torch.zeros_like(T1[rows]), torch.zeros_like(T1[rows])
                    ws = _lib.Workspace(DEV)
                    _lib.infonce_fwd_bwd(T1[rows].contiguous(), T2[rows].contiguous(), idx, tau, 0.05, 0.5, r1, r2,
                                         ref_loss, ws)
                    em = Emulated(nU, nI, world)
                    losses, d1, d2 = infonce_sharded(em, T1, T2, which, idx, D, tau, 0.05, 0.5)
                    what = 'world %d D %d B %d tau %g which %d' % (world, D, B, tau, which)
                    assert len(set(losses)) == 1, what + ': loss bits differ between ranks'
                    assert abs(losses[0] - float(ref_loss[0])) <= 1e-5 * abs(float(ref_loss[0])), what
                    assert_close(host(d1[rows]), host(r1), what + ' dT1', **RED_TOL)
                    assert_close(host(d2[rows]), host(r2), what + ' dT2', **RED_TOL)
                    outside = slice(nU, nU + nI) if which == 0 else slice(0, nU)
                    assert float(d1[outside].abs().max()) == 0.0 and float(d2[outside].abs().max()) == 0.0
                    assert ws.status() == 0 and em.statuses() == [0] * world


@pytest.mark.gpu
@pytest.mark.parametrize('world', WORLDS)
def test_bpr_logsig_sum_sharded_matches_single_gpu(world):
    for si, (nU, nI, B) in enumerate(((2, 203, 1001), (301, 517, 2050))):
        for D in (16, 20, 64):
            U, I = tables(nU, nI, D, 30 + si)
            user, pos, neg = batch(nU, nI, B, 31 + si)
            Ud, Id, ud, pd, nd = dev(U), dev(I), dev(user), dev(pos), dev(neg)
            gU, gI, loss = torch.zeros_like(Ud), torch.zeros_like(Id), torch.zeros(1, device=DEV)
            _lib.bpr_logsig_sum_fwd_bwd(Ud, Id, ud, pd, nd, gU, gI, loss, _lib.Workspace(DEV), grad_scale=0.25)
            em = Emulated(nU, nI, world)
            T = em.structs(em.shards(torch.cat([Ud, Id])))
            G = em.zeros(D)
            Gd = em.structs(G)
            total = 0.0
            for r, lay in enumerate(em.lay):
                lo, hi = lay.batch_slice(B)
                lp = torch.zeros(1, device=DEV)
                _lib.bpr_logsig_sum_fwd_bwd_sharded(T[r], Gd[r], ud[lo:hi], pd[lo:hi], nd[lo:hi], B, D, lp, em.ws[r],
                                                    grad_scale=0.25)
                total += float(lp[0])
            assert abs(total - float(loss[0])) <= 1e-5 * abs(float(loss[0]))
            full = em.full_of(G)
            assert_close(host(full[:nU]), host(gU), 'user gradient', **RED_TOL)
            assert_close(host(full[nU:]), host(gI), 'item gradient', **RED_TOL)
            assert em.statuses() == [0] * world


# ---------------------------------------------------------------------------------------------------------
# GPU: whole SGL steps through model.shard(), emulated ranks
# ---------------------------------------------------------------------------------------------------------

def dense_csr(dense):
    """Host CSR (rows / columns ascending) of a dense matrix -- the order the views' CSRs have."""
    r, c = np.nonzero(dense)
    ptr = np.zeros(dense.shape[0] + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=dense.shape[0]), out=ptr[1:])
    return ptr, c.astype(np.int32), dense[r, c].astype(np.float32)


def check_local_graph(lg, lay, g, what):
    lptr, lcol, lval = host_cut(lay, g)
    nnz = int(lptr[-1])
    assert (host(lg.rowptr) == lptr).all(), what
    assert (host(lg.col[:nnz]) == lcol).all() and host(lg.val[:nnz]).tobytes() == lval.tobytes(), what


def golden_steps_body(tag, peers):
    """One rank of the sharded golden check (emulated or real ranks): the views every rank draws equal the reference's;
    three sharded steps match the goldens with the bars of test_sgl_steps_match_reference_golden (loss, ego gradients
    before Adam, parameters after)."""
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.SGL import SGL
    s = small_case(load('sgl_cases.npz'), tag)
    lr, l2, reg, L, D, tau, w_ssl, drop = (float(x) for x in s['hp'])
    L, D = int(L), int(D)
    nU, nI = s['U0'].shape[0], s['I0'].shape[0]
    tr = s['train'].astype(np.int64)
    corpus = frames_corpus(tr, tr[:1], tr[:1], n_users=nU, n_items=nI)
    args = model_args(SGL, lr=lr, l2=l2, reg_weight=reg, gcn_layers=L, embedding_size=D, ssl_tau=tau, ssl_weight=w_ssl,
                      drop_ratio=drop)
    model = SGL(args, corpus)
    model.load_state_dict({'user_embedding.weight': torch.from_numpy(s['U0']),
                           'item_embedding.weight': torch.from_numpy(s['I0'])})
    model = model.to(peers.device)
    model.fuse()
    model.optimizer = BaseRunner(args)._build_optimizer(model)
    st = model.shard(peers)
    lay = st.layout
    random.seed(1234)                     # every rank's own stream, seeded as init_seed seeds it on every rank
    model.graph_construction()
    for k, name in enumerate(('sub1', 'sub2')):
        fwd, tr_ = model.sharded_sgl.views[k]
        check_local_graph(fwd, lay, dense_csr(s[name]), '%s rank %d' % (name, lay.rank))
        check_local_graph(tr_, lay, dense_csr(s[name].T), '%s transposed rank %d' % (name, lay.rank))
    grad, grad_s = st.symmetric()
    adam = st.adam

    def adam_keeping_the_gradient(*a, **k):
        grad.copy_(st.G)
        return adam(*a, **k)
    st.adam = adam_keeping_the_gradient
    for step in range(3):
        user, pos, neg = (torch.from_numpy(s[f's{step}/{k}'].astype(np.int64)).to(peers.device)
                          for k in ('user', 'pos', 'neg'))
        B = user.numel()
        lo, hi = lay.batch_slice(B)
        loss = model.sharded_train_step(user[lo:hi], pos[lo:hi], neg[lo:hi], B, lr, l2, batch=torch.stack([user, pos, neg]))
        assert_close(float(loss[0]), s[f's{step}/loss'], f'loss step {step}', rtol=5e-6)
        gu, gi = st.gather_full(grad_s)
        # the sharded InfoNCE sums z and Ga per rank, then over the ranks: where Ga_b - t_b cancels, that reordering
        # shows up as a few ulp of the summands, so the ego gradient gets atol_scale 1e-5 (measured: 7.7e-7 on a 0.08
        # gradient at world 3); loss and parameters keep the single-GPU bars
        assert_close(host(gu), s[f's{step}/gU'], f'gU step {step}', rtol=3e-5, atol_scale=1e-5)
        assert_close(host(gi), s[f's{step}/gI'], f'gI step {step}', rtol=3e-5, atol_scale=1e-5)
        for g in [model.sharded_sgl.pool_grad] + [p for p, _ in model.sharded_sgl.view_grad]:
            assert float(g.abs().max()) == 0.0
        u, i = st.gather_full()
        assert_close(host(u), s[f's{step}/U'], f'U step {step}', rtol=3e-5, atol_scale=3e-6)
        assert_close(host(i), s[f's{step}/I'], f'I step {step}', rtol=3e-5, atol_scale=3e-6)
    model.graph_construction()            # the next epoch's views continue every rank's stream
    nnz = model.sharded_sgl.views[0][0].rowptr[-1:].clone()
    peers.dist.all_reduce(nnz, group=peers.group)
    assert int(nnz[0]) == int(s['sub1_epoch2_nnz'])
    st.ws.raise_on_status()
    peers.close()


@pytest.mark.gpu
@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('tag', ['sgl_d16_l2', 'sgl_d32_l3'])
def test_sharded_sgl_steps_match_reference_golden(tag, world):
    run_ranks(world, lambda peers: golden_steps_body(tag, peers))


def sgl_ml100k_epoch(dev, peers=None):
    """One BaseRunner.fit epoch of SGL on ml-100k (seed 3407) and a dev evaluation, on one GPU or sharded over `peers`:
    (per-step losses, dev HR@10 / NDCG@10, parameters after the epoch)."""
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.SGL import SGL
    from whisprrec_b200.utils import utils
    corpus = ml100k_corpus()
    args = model_args(SGL, lr=1e-3, gcn_layers=2, batch_size=1024)
    args.device = dev
    utils.init_seed(3407)
    model = SGL(args, corpus).to(dev)
    model.fuse()
    data = {ph: SGL.Dataset(model, corpus, ph) for ph in ('train', 'dev')}
    runner = BaseRunner(args)
    model.optimizer = runner._build_optimizer(model)
    losses = []
    name = 'predict' if peers is None else 'sharded_train_step'
    if peers is not None:
        model.shard(peers)
    inner = getattr(model, name)

    def recording(*a, **k):
        out = inner(*a, **k)
        losses.append(float(out.reshape(-1)[0]))
        return out
    setattr(model, name, recording)
    runner.fit(data['train'], epoch=1)
    res = runner.evaluate(data['dev'], [10], ['HR', 'NDCG'])
    if peers is None:
        return losses, res, host(model.tables.P)
    u, i = model.sharded.gather_full()
    return losses, res, host(torch.cat([u, i]))


def check_epoch_against_single_gpu(got, ref):
    losses, res, P = got
    ref_losses, ref_res, ref_P = ref
    assert len(losses) == len(ref_losses)
    assert_close(np.array(losses), np.array(ref_losses), 'per-step losses', rtol=1e-4, atol_scale=0.0)
    assert_close(P, ref_P, 'parameters after the epoch', rtol=1e-3, atol_scale=1e-3)
    for k in ('HR@10', 'NDCG@10'):
        assert abs(res[k] - ref_res[k]) <= 1e-3, (k, res[k], ref_res[k])


def ml100k_epoch_body(peers):
    """One rank on real GPUs: the single-GPU epoch on its own device first, then the sharded one."""
    ref = sgl_ml100k_epoch(peers.device)
    check_epoch_against_single_gpu(sgl_ml100k_epoch(peers.device, peers), ref)
    peers.close()


@pytest.mark.gpu
def test_sharded_sgl_ml100k_epoch_matches_single_gpu():
    """One BaseRunner.fit epoch and a dev evaluation at emulated world 2 against the single-GPU epoch, same seeds."""
    ref = sgl_ml100k_epoch(DEV)
    got = [None, None]

    def body(peers):
        got[peers.rank] = sgl_ml100k_epoch(DEV, peers)
        peers.close()
    run_ranks(2, body)
    for g in got:
        check_epoch_against_single_gpu(g, ref)
