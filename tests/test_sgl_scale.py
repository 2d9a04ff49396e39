"""SGL's InfoNCE streamed over the table (wr_infonce_fwd_bwd): no buffer grows with batch x table, so catalogues of any
size train.  CPU: the scratch query has no B x N term, and the argument checks.  GPU: the kernel against the oracle's
InfoNCE under torch autograd (sizes the materialised weight matrix refused, the ml-1m shape, awkward sizes), the same loss
bits from call to call, and SGL end to end on a corpus of 70,000 items."""
import numpy as np
import pytest
import torch

from oracle import whispr_oracle as O
from tests.helpers import assert_close, close, frames_corpus, model_args
from whisprrec_b200 import _lib

DEV = torch.device('cuda:0')


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------

def test_infonce_scratch_has_no_batch_times_table_term():
    q = _lib.load().wr_infonce_scratch_bytes
    for B, N, D in ((2048, 10_000_000, 64), (4096, 2_000_000, 256), (2048, 70_000, 64), (1, 1, 16), (65, 4097, 128),
                    (1_000_000, 3706, 64)):
        # Tn, Gt, An, Ga: 2 (B + N) D floats; per-row scalars; the pass-1 row sums (at most 4 x 148 tiles of 64 rows
        # or one range when the batch alone fills the GPU); the pass-2 Gt partials (only below 2 x 148 table tiles)
        bound = 4 * (2 * (B + N) * D + 2 * N + 3 * B) + 4 * (4 * 148 * 64 + B) + 4 * 7 * 2 * 148 * 64 * D + 12 * 256
        assert 0 < q(B, N, D) <= bound, (B, N, D)
    assert q(2048, 10_000_000, 64) < 6e9 and q(2048, 20_000_000, 64) < 2 * q(2048, 10_000_000, 64)
    assert q(0, 10, 64) == 0 and q(10, 0, 64) == 0 and q(10, 10, 0) == 0 and q(10, 10, 512) == 0


def test_infonce_argument_errors_need_no_gpu():
    lib = _lib.load()
    # wr_infonce_fwd_bwd(T1, T2, idx, B, N, D, tau, weight, grad_scale, dT1, dT2, loss_out, scratch, scratch_bytes, ws,
    #                    stream)
    call = lambda B=8, N=100, D=64, tau=0.1, scratch=16, nbytes=1 << 40, ws=16, t1=16: lib.wr_infonce_fwd_bwd(
        t1, 16, 16, B, N, D, tau, 1.0, 1.0, 16, 16, 16, scratch, nbytes, ws, None)
    assert call(t1=None) == -1 and call(scratch=None) == -1 and call(ws=None) == -1
    assert call(B=0) == -2 and call(N=0) == -2 and call(tau=0.0) == -2 and call(tau=-1.0) == -2
    assert call(D=0) == -3 and call(D=30) == -3
    # D > 256 is refused since InfoNCE is streamed (both operand tiles of pass 2 stay in shared memory); the models
    # and the evaluation kernels stop at 256 too
    assert call(D=260) == -3 and call(D=512) == -3
    assert call(nbytes=lib.wr_infonce_scratch_bytes(8, 100, 64) - 1) == -2
    assert call(B=2048, N=65_537, nbytes=0) == -2


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------

def _oracle_info_nce(T1, T2, idx, tau, weight, grad_scale):
    """sgl_oracle.loss's info_nce (the reference's SGL.py:196-231) on the CPU in fp32; returns (weight * InfoNCE,
    grad_scale * its gradients w.r.t. T1 and T2)."""
    t1 = torch.from_numpy(T1).requires_grad_(True)
    t2 = torch.from_numpy(T2).requires_grad_(True)
    i = torch.from_numpy(idx)
    a = torch.nn.functional.normalize(t1[i], dim=1)
    b = torch.nn.functional.normalize(t2[i], dim=1)
    allb = torch.nn.functional.normalize(t2, dim=1)
    pos_s = torch.exp((a * b).sum(1) / tau)
    tot_s = torch.exp(a.matmul(allb.T) / tau).sum(1)
    val = weight * -torch.sum(torch.log(pos_s / tot_s))
    (val * grad_scale).backward()
    return float(val.detach()), t1.grad.numpy(), t2.grad.numpy()


def _tables(N, D, B, seed, dup=False):
    """Two views with uneven row norms, and batch ids (with repeats when `dup`).  The views are correlated, as SGL's are,
    on tables of 4,096 rows or more.  On smaller ones they are independent: with a handful of rows and a dominant
    positive pair, log z_b - s_b cancels down to the fp32 rounding of s_b itself, in the oracle as in any fp32 kernel."""
    rng = np.random.RandomState(seed)
    T1 = (rng.randn(N, D) * rng.uniform(0.1, 2.0, (N, 1))).astype(np.float32)
    noise = rng.randn(N, D).astype(np.float32)
    T2 = (T1 + 0.5 * noise if N >= 4096 else noise).astype(np.float32)
    idx = rng.randint(0, N, B).astype(np.int64)
    if dup and B > 4:
        idx[1] = idx[0]
        idx[B // 2:B // 2 + 3] = idx[2]
    return T1, T2, idx


def _run(T1, T2, idx, tau, weight, grad_scale, ws):
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    t1, t2, ix = d(T1), d(T2), d(idx)
    g1, g2 = torch.zeros_like(t1), torch.zeros_like(t2)
    loss = torch.zeros(1, device=DEV)
    _lib.infonce_fwd_bwd(t1, t2, ix, tau, weight, grad_scale, g1, g2, loss, ws)
    return float(loss.item()), g1.cpu().numpy(), g2.cpu().numpy()


@pytest.fixture(scope='module')
def ws():
    return _lib.Workspace(DEV)


@pytest.mark.gpu
@pytest.mark.parametrize('B,N,D,tau,weight,grad_scale,dup', [
    (2048, 70_000, 64, 0.1, 0.05, 1 / 3, False),        # refused by the materialised path
    (4096, 40_000, 32, 0.1, 0.05, 1 / 3, False),        # refused by the materialised path
    (2048, 65_537, 64, 0.1, 1.0, 1.0, True),            # one past the materialised path's last size
    (2048, 6040, 64, 0.1, 0.05, 1 / 3, False),          # ml-1m users
    (2048, 3706, 64, 0.1, 0.05, 1 / 3, True),           # ml-1m items
    (1, 1, 16, 0.1, 1.0, 1.0, False),
    (1, 4097, 128, 0.5, 2.0, 0.25, False),
    (65, 63, 256, 0.1, 0.05, 0.5, True),
    (65, 4097, 16, 0.5, 1.0, 1.0, True),
    (65, 1, 128, 0.5, 0.3, 1.0, True),
    (1, 63, 256, 0.1, 1.0, 1.0, False),
    (4096, 12_000, 256, 0.5, 0.05, 1 / 3, False),       # two batch ranges in pass 2 at the largest D
    (65, 4097, 20, 0.1, 0.05, 1 / 3, True),             # D padded to 32 (two-column groups, columns past D masked)
    (130, 300, 68, 0.5, 1.0, 0.5, False),               # D padded to 128
    (600, 5000, 36, 0.1, 0.05, 1 / 3, True),            # 10 batch tiles: rotated start, padded D
])
def test_infonce_matches_the_oracle(B, N, D, tau, weight, grad_scale, dup, ws):
    T1, T2, idx = _tables(N, D, B, seed=B + N + D, dup=dup)
    o_loss, o_g1, o_g2 = _oracle_info_nce(T1, T2, idx, tau, weight, grad_scale)
    loss, g1, g2 = _run(T1, T2, idx, tau, weight, grad_scale, ws)
    assert ws.status() == 0
    if N == 1:
        # one table row: every row's softmax is exactly 1, so the loss and the gradients are 0 up to rounding
        inv = 1.0 / min(np.linalg.norm(T1, axis=1).min(), np.linalg.norm(T2, axis=1).min())
        assert abs(loss - o_loss) <= 1e-6 * weight * B / tau
        for g, o in ((g1, o_g1), (g2, o_g2)):
            assert np.abs(g - o).max() <= 1e-5 * weight * grad_scale / tau * inv * B
        return
    assert loss == pytest.approx(o_loss, rel=1e-5)
    assert_close(g1, o_g1, 'dT1')
    assert_close(g2, o_g2, 'dT2')


@pytest.mark.gpu
def test_infonce_loss_has_the_same_bits_from_call_to_call(ws):
    T1, T2, idx = _tables(70_000, 64, 2048, seed=5, dup=True)
    a, b = _run(T1, T2, idx, 0.1, 0.05, 1 / 3, ws), _run(T1, T2, idx, 0.1, 0.05, 1 / 3, ws)
    assert np.float32(a[0]).tobytes() == np.float32(b[0]).tobytes()
    assert ws.status() == 0


def _large_catalogue_corpus():
    """5,000 users x 70,000 items (more than the 65,536 the materialised path took at batch 2048), power-law."""
    from whisprrec_b200.utils import synthetic
    nU, nI = 5000, 70_000
    u, i = synthetic.power_law_pairs(nU, nI, 120_000, seed=11)
    pairs = np.stack([u.numpy(), i.numpy()], 1)
    rng = np.random.RandomState(0)
    pairs = pairs[rng.permutation(len(pairs))]
    _, first = np.unique(pairs[:, 0], return_index=True)
    dev = pairs[first[:1000]]
    train = np.delete(pairs, first[:1000], axis=0)
    return frames_corpus(train, dev, dev[:1], n_users=nU, n_items=nI)


@pytest.fixture(scope='module')
def big_corpus():
    return _large_catalogue_corpus()


@pytest.mark.gpu
def test_sgl_steps_on_70000_items_match_the_oracle(big_corpus):
    """Three predict + FusedAdam steps against sgl_oracle.fwd_bwd + Adam.  As in the ml-100k two-epoch test, Adam's
    m / sqrt(v) can turn a last-bit difference of a near-zero InfoNCE gradient into a step of up to lr, so a few
    parameters in 10^5 may differ by that much."""
    from oracle import sgl_oracle as SO
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.SGL import SGL
    from whisprrec_b200.utils import utils
    corpus = big_corpus
    nU, nI = corpus.n_users, corpus.n_items
    args = model_args(SGL, lr=1e-3, l2=0.0)
    utils.init_seed(3407)
    model = SGL(args, corpus).to(DEV)
    t = model.fuse()
    model.optimizer = BaseRunner(args)._build_optimizer(model)
    model.graph_construction()
    host = lambda x: x.detach().cpu().numpy()
    graphs = [O.csr_to_torch(host(g.rowptr), host(g.col), host(g.val), nU + nI)
              for g in [model.train_graph] + model.sub_graphs]
    oU, oI = torch.from_numpy(host(t.P[:nU]).copy()), torch.from_numpy(host(t.P[nU:]).copy())
    om = [torch.zeros_like(oU), torch.zeros_like(oU), torch.zeros_like(oI), torch.zeros_like(oI)]
    tr = corpus.data_df['train']
    rng = np.random.RandomState(1)
    for step in range(1, 4):
        sel = rng.randint(0, len(tr), args.batch_size)
        user = tr['user_id'].values[sel].astype(np.int64)
        pos = tr['item_id'].values[sel].astype(np.int64)
        neg = rng.randint(0, nI, args.batch_size).astype(np.int64)
        d = lambda a: torch.from_numpy(a).to(DEV)
        loss = model.predict({'user_id': d(user), 'pos_item': d(pos), 'neg_items': d(neg)})
        o_loss, gU, gI = SO.fwd_bwd(oU.numpy(), oI.numpy(), graphs, user, pos, neg, model.gcn_layers, model.reg_weight,
                                    model.ssl_tau, model.ssl_weight)
        assert float(loss) == pytest.approx(float(o_loss), rel=1e-4), step
        model.optimizer.step()
        O.adam_l2_step(oU, om[0], om[1], gU, step, args.lr, args.l2)
        O.adam_l2_step(oI, om[2], om[3], gI, step, args.lr, args.l2)
    for what, got, want in (('U', host(t.P[:nU]), oU.numpy()), ('I', host(t.P[nU:]), oI.numpy())):
        off = ~close(got, want, 1e-3, 1e-3)
        assert off.mean() <= 1e-5 and np.abs(got - want).max() <= 2 * args.lr, (what, off.sum())
    assert t.ws.status() == 0


@pytest.mark.gpu
def test_sgl_epoch_on_70000_items_runs_through_the_runner(big_corpus):
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.SGL import SGL
    from whisprrec_b200.utils import utils
    args = model_args(SGL, lr=1e-3, l2=0.0)
    utils.init_seed(3407)
    model = SGL(args, big_corpus).to(DEV)
    model.fuse()
    runner = BaseRunner(args)
    model.optimizer = runner._build_optimizer(model)
    data = {ph: SGL.Dataset(model, big_corpus, ph) for ph in ('train', 'dev')}
    mean_loss = runner.fit(data['train'], epoch=1)
    res = runner.evaluate(data['dev'], [10, 20], ['NDCG', 'HR'])
    assert np.isfinite(mean_loss) and 0.0 <= res['HR@20'] <= 1.0
    assert model.tables.ws.status() == 0
