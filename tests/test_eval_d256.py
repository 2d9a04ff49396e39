"""Full-ranking evaluation at embedding size 256: the fp32 FMA tiles (precision 0), the bf16 tensor-core path (1) and the
split-bf16 tensor-core path with the exact re-check (2), from the kernels up to BaseRunner, on the shapes the D <= 128
tests use."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import whispr_oracle as O
from tests.helpers import assert_close, close, ml100k_corpus, model_args
from whisprrec_b200 import _lib
from whisprrec_b200.models.general.BPRMF import BPRMF
from whisprrec_b200.models.general.LightGCN import LightGCN
from whisprrec_b200.models.general.SGL import SGL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D = 256
DEV = torch.device('cuda:0')


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------

def test_models_accept_256_and_still_refuse_other_sizes():
    corpus = ml100k_corpus()
    for cls in (BPRMF, LightGCN, SGL):
        assert cls(model_args(cls, embedding_size=256), corpus).emb_size == 256
        for bad in (96, 512):
            with pytest.raises(ValueError, match='embedding_size'):
                cls(model_args(cls, embedding_size=bad), corpus)
    assert 256 in _lib.EVAL_DIMS


def test_exact_tensor_core_path_covers_256():
    assert _lib.exact_tc_supported(256)
    assert not _lib.exact_tc_supported(256, k=10) and not _lib.exact_tc_supported(256, scores=True)


def test_scratch_holds_the_hi_lo_resident_layout():
    """precision 2 at D = 256 keeps the user rows as [hi | lo] (2 D bf16) and the items as [hi | lo | hi] (3 D bf16)."""
    lib = _lib.load()
    for R, n in ((1000, 5000), (262_144, 1_000_000), (1, 10)):
        need = R * 2 * D * 2 + n * 3 * D * 2 + R + R * 4
        assert lib.wr_eval_scratch_bytes(R, n, D, 2) >= need
        assert lib.wr_eval_scratch_bytes(R, n, D, 1) >= (R + n) * D * 2 + R


def test_exact_band_at_256_has_margin():
    """c_256 = 3.1e-4: the three-term split-bf16 sum stays an order of magnitude inside the band (float64)."""
    rng = np.random.RandomState(0)
    c = 3.1e-4
    a = (rng.randn(2000, D) * rng.uniform(0.01, 10, (2000, 1))).astype(np.float32)
    b = (rng.randn(2000, D) * rng.uniform(0.01, 10, (2000, 1))).astype(np.float32)
    bf = lambda x: (torch.from_numpy(x).to(torch.bfloat16).to(torch.float32)).numpy()
    ah, bh = bf(a), bf(b)
    al, bl = bf(a - ah), bf(b - bh)
    three = (ah.astype(np.float64) * bh + ah.astype(np.float64) * bl + al.astype(np.float64) * bh).sum(1)
    exact = (a.astype(np.float64) * b).sum(1)
    scale = np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1)
    assert (np.abs(three - exact) / scale).max() < c / 10
    # the derivation of DESIGN.md section 4.3: twice (lo.lo residual + fp32 sum of 3 D products + precision 0's chain)
    assert 2 * (3.1 * 2.0 ** -16 + 3 * D * 2.0 ** -23 + D * 2.0 ** -24) <= c


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------

def dv(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host(t):
    return t.detach().cpu().numpy()


@pytest.fixture
def ws():
    w = _lib.Workspace(DEV)
    yield w
    assert w.status() == 0


def problem(R, nI, seed, hmax, scale_u=1.0):
    rng = np.random.RandomState(seed)
    nU = max(2, R // 3)
    U = (rng.randn(nU, D) * scale_u).astype(np.float32)
    I = rng.randn(nI, D).astype(np.float32)
    user = rng.randint(0, nU, R).astype(np.int64)
    pos = rng.randint(0, nI, R).astype(np.int64)
    hist = [np.sort(rng.choice(nI, size=min(nI, rng.randint(0, hmax)), replace=False)) for _ in range(nU)]
    hist[0] = np.arange(nI)                                   # a user who has seen everything
    hist[1] = np.zeros(0, dtype=np.int64)                     # and one with no history
    hp = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum([len(h) for h in hist], out=hp[1:])
    hi = np.concatenate(hist + [np.zeros(1)]).astype(np.int32)
    return U, I, user, pos, hp, hi


@pytest.mark.gpu
@pytest.mark.parametrize('R,nI', [(1, 10), (65, 64), (300, 129), (3000, 5000), (500, 1000)])
def test_fp32_eval_at_256_vs_oracle_and_self_consistency(R, nI, ws):
    """Ragged tiles, users with no / full history, splits of the item range, k = 1..32, the dense score dump and the
    item-shard entry point (one shard = the whole table)."""
    U, I, user, pos, hp, hi = problem(R, nI, R + nI + D, 40)
    k = min(32, nI)
    for want_topk in (0, 1, k):
        rank, target, tki, tkv, scores = _lib.eval_rank_topk(dv(U), dv(I), dv(user), dv(pos), dv(hp), dv(hi), ws,
                                                             k=want_topk, scores=True)
        sc = host(scores)
        o_scores = O.full_scores(U, I, user).numpy()
        assert_close(sc, o_scores, 'scores', rtol=1e-5, atol_scale=2e-6)
        o_rank, _ = O.ranks_count(o_scores, user, pos, hp, hi)
        assert np.mean(host(rank) != o_rank) <= 2e-3
        s_rank, s_target = O.ranks_count(sc, user, pos, hp, hi)
        assert (host(rank) == s_rank).all()
        assert (host(target) == s_target).all()
        if want_topk:
            ref_idx, ref_val = O.topk_masked(sc, user, hp, hi, want_topk)
            got_idx, got_val = host(tki), host(tkv)
            filled = np.isfinite(ref_val)
            assert (got_idx[filled] == ref_idx[filled]).all()
            assert (got_val[filled] == ref_val[filled]).all()
            assert (got_idx[~filled] == -1).all() and np.isneginf(got_val[~filled]).all()
        # item-shard mode: gathered user rows, the target as an input
        rank_s, tki_s, tkv_s = _lib.eval_rank_topk_shard(dv(U[user]), dv(I), dv(user), dv(pos), U.shape[0], dv(hp),
                                                         dv(hi), target, ws, k=want_topk)
        assert torch.equal(rank_s, rank)
        if want_topk:
            assert torch.equal(tki_s, tki) and torch.equal(tkv_s, tkv)
        # without the score dump (the production call) nothing changes
        rank2, target2, tki2, tkv2, _ = _lib.eval_rank_topk(dv(U), dv(I), dv(user), dv(pos), dv(hp), dv(hi), ws,
                                                            k=want_topk)
        assert torch.equal(rank2, rank) and torch.equal(target2, target)
        if want_topk:
            assert torch.equal(tki2, tki) and torch.equal(tkv2, tkv)


def check_bf16_path(R, nI, ws):
    """precision 1 against the bf16-rounded oracle at the tolerances of the D <= 128 test; top-k exact against the
    kernel's own scores."""
    U, I, user, pos, hp, hi = problem(R, nI, R + nI + D, 60, scale_u=1.0 / np.sqrt(D))
    rank, target, _, _, scores = _lib.eval_rank_topk(dv(U), dv(I), dv(user), dv(pos), dv(hp), dv(hi), ws,
                                                     precision=1, scores=True)
    o_scores = O.full_scores_bf16(U, I, user).numpy()
    assert_close(host(scores), o_scores, 'tensor-core scores', rtol=2e-5, atol_scale=4e-6)
    assert_close(host(target), o_scores[np.arange(R), pos], 'target', rtol=2e-5, atol_scale=4e-6)
    sc, tg = host(scores), host(target)
    gt = sc > tg[:, None]
    gt[np.arange(R), pos] = False
    for r_, u_ in enumerate(user):
        gt[r_, hi[hp[u_]:hp[u_ + 1]]] = False
    assert (host(rank) == 1 + gt.sum(1)).all()
    o_rank, _ = O.ranks_count(o_scores, user, pos, hp, hi)
    assert np.mean(host(rank) != o_rank) <= 5e-3
    rank2 = _lib.eval_rank_topk(dv(U), dv(I), dv(user), dv(pos), dv(hp), dv(hi), ws, precision=1)[0]
    assert torch.equal(rank, rank2)
    for k in (10, 32):
        rank3, _, tki, tkv, _ = _lib.eval_rank_topk(dv(U), dv(I), dv(user), dv(pos), dv(hp), dv(hi), ws, k=k,
                                                    precision=1)
        assert torch.equal(rank, rank3)
        want_i, want_v = O.topk_masked(sc, user, hp, hi, k)
        want_i = np.where(np.isfinite(want_v), want_i, -1)
        want_i[:, nI:] = -1
        got_i, got_v = host(tki), host(tkv)
        kk = min(k, nI)
        assert (got_i[:, :kk] == want_i[:, :kk]).all(), f'top-{k} ids'
        assert (got_v[:, :kk][want_i[:, :kk] >= 0] == want_v[:, :kk][want_i[:, :kk] >= 0]).all(), f'top-{k} values'
        assert (got_i[:, kk:] == -1).all()
    assert ws.status() == 0


@pytest.mark.gpu
@pytest.mark.parametrize('R,nI', [(128, 256), (130, 700), (3000, 5000), (500, 1000), (1, 10)])
def test_bf16_tensor_core_eval_at_256_vs_bf16_oracle(R, nI, ws):
    check_bf16_path(R, nI, ws)


@pytest.mark.gpu
def test_bf16_tensor_core_eval_at_256_other_layouts():
    """The per-thread top-k lists (WR_TC_TOPK_MODE=1) and the 256-row CTA (WR_TC_VARIANT=12); the library reads both
    switches once per process, hence the child process."""
    code = ('import torch; from whisprrec_b200 import _lib; from tests import test_eval_d256 as t\n'
            'ws = _lib.Workspace(torch.device("cuda:0"))\n'
            'for R, nI in ((130, 700), (3000, 5000)): t.check_bf16_path(R, nI, ws)\n'
            'print("bf16 layouts ok")\n')
    env = dict(os.environ, WR_TC_TOPK_MODE='1', WR_TC_VARIANT='12')
    r = subprocess.run([sys.executable, '-c', code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'bf16 layouts ok' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize('R,nI', [(3000, 40_000), (2500, 33_333), (257, 300), (90_000, 5_000)])
def test_exact_tensor_core_eval_at_256_equals_the_fp32_path(R, nI, ws):
    """precision 2 against precision 0 on the adversarial tables of the D <= 128 test: item norms spread over 3x, exact
    ties, an all-zero user, long histories.  Ranks and target scores identical, no candidate-list overflow; the item-shard
    entry point too."""
    rng = np.random.RandomState(D + R)
    nU = 5000
    U = (rng.randn(nU, D) / np.sqrt(D)).astype(np.float32)
    I = (rng.randn(nI, D) * rng.uniform(0.5, 1.5, (nI, 1))).astype(np.float32)
    I[7] = I[3]
    I[nI - 1] = I[nI - 2]
    U[11] = 0.0
    user = rng.randint(0, nU, R).astype(np.int64)
    user[:4] = 11
    pos = rng.randint(0, nI, R).astype(np.int64)
    pos[5], pos[6] = 3, 7
    hl = rng.randint(0, 60, nU)
    hptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(hl, out=hptr[1:])
    hidx = np.concatenate([np.sort(rng.choice(nI, n, replace=False)) for n in hl]).astype(np.int32)
    dU, dI, du, dp, dh, di = dv(U), dv(I), dv(user), dv(pos), dv(hptr), dv(hidx)
    r0, t0, _, _, _ = _lib.eval_rank_topk(dU, dI, du, dp, dh, di, ws, precision=0)
    r2, t2, _, _, _ = _lib.eval_rank_topk(dU, dI, du, dp, dh, di, ws, precision=2)
    assert ws.status() == 0, 'candidate list overflow'
    assert torch.equal(t0, t2), 'target scores'
    bad = (r0 != r2).nonzero().flatten()
    assert bad.numel() == 0, ('ranks differ', bad[:8].tolist(), r0[bad[:8]].tolist(), r2[bad[:8]].tolist())
    rs = _lib.eval_rank_topk_shard(dv(U[user]), dI, du, dp, nU, dh, di, t0, ws, precision=2)[0]
    assert ws.status() == 0
    assert torch.equal(rs, r0), 'item-shard entry point'


# ---- end to end: ml-100k through BaseRunner, against the oracle ----

def _oracle_epochs(cls, model, args, corpus, epochs):
    """Run `epochs` epochs through BaseRunner.fit and the same batches through the oracle (Adam with L2 as the fused
    models apply it); returns (mean losses, oracle mean losses, model, runner, data, oracle U, oracle I)."""
    from oracle import sgl_oracle as SO
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    t = model.fuse()
    nU = corpus.n_users
    runner = BaseRunner(args)
    model.optimizer = runner._build_optimizer(model)
    data = {ph: cls.Dataset(model, corpus, ph) for ph in ('train', 'dev')}
    oU, oI = torch.from_numpy(host(t.P[:nU]).copy()), torch.from_numpy(host(t.P[nU:]).copy())
    om = [torch.zeros_like(oU), torch.zeros_like(oU), torch.zeros_like(oI), torch.zeros_like(oI)]
    captured = []
    batches_of = runner.epoch_batches

    def capture(dataset):
        b = batches_of(dataset)
        captured.append(host(b))
        return b
    runner.epoch_batches = capture
    if cls is LightGCN:
        ptr, idx = corpus.train_csr()
        tu = np.repeat(np.arange(nU), np.diff(ptr))
        rowptr, col, val = O.build_norm_adj_csr(nU, corpus.n_items, tu, np.asarray(idx))
        A = O.csr_to_torch(rowptr, col, val, nU + corpus.n_items)
    got, want, step = [], [], 0
    for _ in range(epochs):
        got.append(runner.fit(data['train'], epoch=1))
        b = captured[-1]
        if cls is SGL:
            N = nU + corpus.n_items
            graphs = [O.csr_to_torch(host(g.rowptr), host(g.col), host(g.val), N)
                      for g in [model.train_graph] + model.sub_graphs]
        losses = []
        for lo in range(0, b.shape[1], args.batch_size):
            user, pos, neg = (b[j, lo:lo + args.batch_size] for j in range(3))
            if cls is BPRMF:
                loss, gU, gI = O.bpr_fwd_bwd(oU, oI, user, pos, neg)
            elif cls is LightGCN:
                loss, gU, gI = O.lightgcn_fwd_bwd(A, oU, oI, user, pos, neg, model.gcn_layers, model.reg_weight)
            else:
                loss, gU, gI = SO.fwd_bwd(oU.numpy(), oI.numpy(), graphs, user, pos, neg, model.gcn_layers,
                                          model.reg_weight, model.ssl_tau, model.ssl_weight)
            step += 1
            O.adam_l2_step(oU, om[0], om[1], gU, step, args.lr, args.l2)
            O.adam_l2_step(oI, om[2], om[3], gI, step, args.lr, args.l2)
            losses.append(float(loss))
        want.append(float(np.mean(losses)))
    runner.epoch_batches = batches_of
    return got, want, runner, data, oU, oI


@pytest.mark.gpu
@pytest.mark.parametrize('cls,over,loss_rtol,tol,outliers', [
    (BPRMF, dict(lr=1e-3, l2=1e-6), 1e-5, 1e-4, 0.0),
    (LightGCN, dict(lr=2e-3, gcn_layers=2), 1e-4, 1e-3, 0.0),
    (SGL, dict(lr=1e-3, l2=0.0), 1e-4, 1e-3, 1e-5),
])
def test_ml100k_two_epochs_at_256_match_the_oracle(cls, over, loss_rtol, tol, outliers):
    """`--embedding_size 256` end to end: two epochs of BaseRunner.fit against the oracle on the same batches, then the
    dev metrics of the exact tensor-core evaluation (the runner's default) equal those of the fp32 path bit for bit.
    SGL: Adam's m / sqrt(v) turns a last-bit difference of a near-zero InfoNCE gradient (fp32 FMA tiles against the
    oracle's autograd) into up to a whole step of size lr, so a few parameters in 10^5 may differ by that much."""
    from whisprrec_b200.utils import utils
    corpus = ml100k_corpus()
    args = model_args(cls, embedding_size=D, **over)
    utils.init_seed(3407)
    model = cls(args, corpus).to(DEV)
    got, want, runner, data, oU, oI = _oracle_epochs(cls, model, args, corpus, 2)
    for g_, w_ in zip(got, want):
        assert g_ == pytest.approx(w_, rel=loss_rtol), (got, want)
    ue, ie = model._embedding_pair()
    for what, got_p, want_p in (('U', host(ue.weight), oU.numpy()), ('I', host(ie.weight), oI.numpy())):
        if outliers:
            off = ~close(got_p, want_p, tol, tol)
            assert off.mean() <= outliers and np.abs(got_p - want_p).max() <= 2 * args.lr, (what, off.sum())
        else:
            assert_close(got_p, want_p, what + ' after two epochs', rtol=tol, atol_scale=tol)
    assert runner.eval_precision == 2
    ws = model.tables.ws
    res2 = runner.evaluate(data['dev'], [5, 10, 20], ['NDCG', 'HR'])
    assert ws.status() == 0
    runner.eval_precision = 0
    res0 = runner.evaluate(data['dev'], [5, 10, 20], ['NDCG', 'HR'])
    assert res2 == res0
    assert 0.0 < res0['HR@20'] < 1.0
