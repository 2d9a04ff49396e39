"""Top-k lists at precision 2: precision 0's lists (same ids, same fp32 values, same order) from the split-bf16 tensor-core
path.  CPU: the support predicate, argument errors, the scratch query, the band's margin for |t - s| and a NumPy model of
the candidate rule.  GPU: identity with precision 0 on adversarial tables, the per-row fallback, emulated item shards and
ml-100k models through BaseRunner."""
import numpy as np
import pytest
import torch

from tests.helpers import ml100k_corpus, model_args
from whisprrec_b200 import _lib

DEV = torch.device('cuda:0')
BAND_C = {64: 1.5e-4, 128: 2.0e-4, 256: 3.1e-4}


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------

def test_exact_topk_support_truth_table():
    for D in (16, 32, 64, 128, 256, 512):
        for k in (0, 1, 10, 32, 33):
            for scores in (False, True):
                want = D in (64, 128, 256) and 1 <= k <= 32 and not scores
                assert _lib.exact_tc_topk_supported(D, k, scores) == want, (D, k, scores)
    # the ranks-only predicate is unchanged
    assert _lib.exact_tc_supported(128) and not _lib.exact_tc_supported(128, k=10)


def test_exact_topk_argument_errors_need_no_gpu():
    lib = _lib.load()
    # wr_eval_rank_topk(U, I, user, pos, R, n_users, n_items, D, hist_ptr, hist_idx, k, precision, topk_idx, topk_val,
    #                   rank, target, scores_out, scratch, ws, stream)
    call = lambda D, k, tk, scores=None, scratch=1024: lib.wr_eval_rank_topk(
        16, 16, 16, 16, 4, 4, 4, D, 16, 16, k, 2, tk, tk, 16, 16, scores, scratch, 16, None)
    assert call(64, 33, 16) == -4
    assert call(64, 0, 16) == -4
    assert call(32, 10, 16) == -3                      # no tensor-core path at D = 32
    assert call(16, 10, 16) == -3
    assert call(64, 10, 16, scratch=None) == -1
    assert call(64, 10, 16, scores=16) == -4           # no dense score dump at precision 2
    assert lib.wr_eval_rank_topk(16, 16, 16, 16, 4, 4, 4, 64, 16, 16, 10, 2, 16, None, 16, 16, None, 1024, 16,
                                 None) == -1           # one of the two list outputs missing
    # wr_eval_rank_topk_shard(Urows, I, user, pos_local, R, n_users, n_items, D, hist_ptr, hist_idx, k, precision,
    #                         target, topk_idx, topk_val, rank, scratch, ws, stream)
    shard = lambda D, k, scratch=1024: lib.wr_eval_rank_topk_shard(16, 16, 16, 16, 4, 4, 4, D, 16, 16, k, 2, 16, 16, 16,
                                                                   16, scratch, 16, None)
    assert shard(64, 33) == -4 and shard(32, 10) == -3 and shard(256, 10, None) == -1
    assert lib.wr_eval_rank_topk_shard(16, 16, 16, 16, 4, 4, 4, 64, 16, 16, 10, 2, None, 16, 16, 16, 1024, 16,
                                       None) == -1


def test_exact_topk_scratch_query():
    lib = _lib.load()
    for R, n in ((1, 10), (3000, 40_000), (90_000, 5_000), (262_144, 1_000_000), (1_000_000, 1_000)):
        for D in (64, 128, 256):
            old = lib.wr_eval_scratch_bytes(R, n, D, 2)
            assert lib.wr_eval_scratch_bytes_topk(R, n, D, 2, 0) == old
            assert lib.wr_eval_scratch_bytes_topk(R, n, D, 1, 10) == lib.wr_eval_scratch_bytes(R, n, D, 1)
            assert lib.wr_eval_scratch_bytes_topk(R, n, D, 0, 10) == 0
            # one row block's segments (1,024 ids and a count per row): the rank path's blocks of ~16e9 / n_items
            # rows, at most 262,144 so that they stay <= 1 GB
            rows = max(256, int(16e9 / n) // 256 * 256)
            if rows > R:
                rows = (R + 255) // 256 * 256
            rows = min(rows, 262_144)
            for k in (1, 10, 32):
                got = lib.wr_eval_scratch_bytes_topk(R, n, D, 2, k)
                assert old + rows * 1024 * 4 + rows * 4 <= got <= old + rows * 1024 * 4 + rows * 4 + 3072
                assert got - old <= (1 << 30) + (1 << 21)
    # the rank-only query itself: bf16 copies + row flags + norms + candidate list (as before)
    assert lib.wr_eval_scratch_bytes(1000, 5000, 64, 2) >= 1000 * 3 * 64 * 2 + 5000 * 3 * 64 * 2 + 1000 + 4000


def _fp32_chain(a, b):
    """precision 0's score: s = fmaf(a_d, b_d, s), d = 0 .. D-1 (the float64 product of two floats is exact)."""
    s = np.zeros(a.shape[0], dtype=np.float32)
    for d in range(a.shape[1]):
        s = (a[:, d].astype(np.float64) * b[:, d] + s).astype(np.float32)
    return s


def _split_bf16(x):
    hi = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    lo = torch.from_numpy(x - hi).to(torch.bfloat16).to(torch.float32).numpy()
    return hi, lo


def _three_term_fp32(a, b):
    """The tensor-core score modelled: hi.hi + hi.lo + lo.hi, the 3 D exact products summed in fp32."""
    ah, al = _split_bf16(a)
    bh, bl = _split_bf16(b)
    t = np.zeros(a.shape[0], dtype=np.float32)
    for x, y in ((ah, bh), (ah, bl), (al, bh)):
        for d in range(a.shape[1]):
            t = (t + (x[:, d].astype(np.float64) * y[:, d]).astype(np.float32)).astype(np.float32)
    return t


@pytest.mark.parametrize('D', [64, 128, 256])
def test_exact_topk_band_bounds_every_score_with_margin(D):
    """The list rule needs |t_j - s_j| <= eps_r / 2 (eps_r = c_D ||a_r|| max ||b||) for EVERY item, with t the fp32
    tensor-core score itself.  c_D is about twice (split residual + fp32 sum of 3 D products + precision 0's chain);
    measured in float64 on fp32-modelled t and s the error stays well inside half of it."""
    c = BAND_C[D]
    # the worst case of |t - s| / (||a|| ||b||) is below c_D / 1.98 (c_128 = 2e-4 rounds 2 x 1.007e-4 down): eps_r bounds
    # |t - s| with room to spare for the rounding of tau - 2 eps_r
    assert 1.98 * (3.1 * 2.0 ** -16 + 3 * D * 2.0 ** -23 + D * 2.0 ** -24) <= c
    rng = np.random.RandomState(D)
    n = 1500
    a = (rng.randn(n, D) * rng.uniform(0.01, 10, (n, 1))).astype(np.float32)
    b = (rng.randn(n, D) * rng.uniform(0.01, 10, (n, 1))).astype(np.float32)
    b[:100] = np.abs(b[:100])                          # same-sign products: no cancellation to hide the rounding
    a[:100] = np.abs(a[:100])
    t, s = _three_term_fp32(a, b), _fp32_chain(a, b)
    scale = np.linalg.norm(a.astype(np.float64), axis=1) * np.linalg.norm(b.astype(np.float64), axis=1)
    err = np.abs(t.astype(np.float64) - s) / scale
    assert err.max() < c / 2 / 4, err.max()


def _top_worse(v, i, w, wi):
    return v < w or (v == w and i > wi)


def _candidates(t, eps, k):
    """The drain warps' rule on one row, scores in item order: the running k-best list over t, tau = its k-th best;
    an item is kept when it enters the list or (eps > 0) t_j >= tau_on_arrival - 2 eps (rounded as the kernel rounds)."""
    lv, li, out = [], [], []
    for j, x in enumerate(t):
        x = np.float32(x)
        if not np.isfinite(x):
            continue
        if len(lv) < k:
            lv.append(x), li.append(j), out.append(j)
            continue
        wp = max(range(k), key=lambda q: (-lv[q], li[q]))   # the worst kept entry
        w, wid = lv[wp], li[wp]
        if _top_worse(w, wid, x, j):
            lv[wp], li[wp] = x, j
            out.append(j)
        elif eps > 0 and x >= np.float32(w - np.float32(np.float32(2 * eps) + np.float32(2.4e-7) * np.float32(abs(w)))):
            out.append(j)
    return set(out)


def _exact_topk(s, k):
    order = sorted((j for j in range(len(s)) if np.isfinite(s[j])), key=lambda j: (-s[j], j))
    return order[:k]


def test_exact_topk_candidate_rule_keeps_the_exact_lists():
    """The candidate set built from the tensor-core scores contains precision 0's top k: random rows, rows with many
    ties (duplicated items, coarse values), an all-zero user row (eps = 0: the first k items, ties by id)."""
    rng = np.random.RandomState(1)
    D, n = 64, 3000
    I = (rng.randn(n, D) * rng.uniform(0.5, 1.5, (n, 1))).astype(np.float32)
    I[n // 2:n // 2 + 200] = I[10]                    # 200 duplicates of one item
    I[2000:2100] = np.round(I[2000:2100])
    bmax = np.linalg.norm(I.astype(np.float64), axis=1).max() * 1.000001
    users = [(rng.randn(D) / 8).astype(np.float32) for _ in range(6)]
    users.append(np.round(rng.randn(D)).astype(np.float32))
    users.append(I[10] * np.float32(0.5))             # the duplicated item is this user's best
    users.append(np.zeros(D, dtype=np.float32))
    for u in users:
        A = np.repeat(u[None], n, 0)
        t, s = _three_term_fp32(A, I), _fp32_chain(A, I)
        s[rng.choice(n, 40, replace=False)] = -np.inf     # history
        t[~np.isfinite(s)] = -np.inf
        eps = BAND_C[D] * np.linalg.norm(u.astype(np.float64)) * 1.000001 * bmax
        for k in (1, 10, 32):
            cand = _candidates(t, eps, k)
            want = _exact_topk(s, k)
            assert set(want) <= cand, (k, sorted(set(want) - cand))
            if eps == 0:                              # the all-zero row: only list entries, ties by id
                assert cand == set(want)
            got = sorted(cand, key=lambda j: (-s[j], j))[:k]
            assert got == want


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------

def dv(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture
def ws():
    w = _lib.Workspace(DEV)
    yield w
    assert w.status() == 0


def adversarial(D, R, nI, seed):
    """The tables of the precision-2 rank tests: item norms over 3x, duplicated items, an all-zero user, long
    histories; plus a user whose history leaves only three items (fewer than k)."""
    rng = np.random.RandomState(seed)
    nU = 5000
    U = (rng.randn(nU, D) / np.sqrt(D)).astype(np.float32)
    I = (rng.randn(nI, D) * rng.uniform(0.5, 1.5, (nI, 1))).astype(np.float32)
    if nI > 7:
        I[7] = I[3]
    I[nI - 1] = I[nI - 2]
    U[11] = 0.0
    user = rng.randint(0, nU, R).astype(np.int64)
    user[:min(R, 4)] = 11
    if R > 8:
        user[8] = 12
    pos = rng.randint(0, nI, R).astype(np.int64)
    if R > 6:
        pos[5], pos[6] = min(3, nI - 1), min(7, nI - 1)
    hl = rng.randint(0, min(60, nI), nU)
    hl[12] = max(0, nI - 3)
    hist = [np.sort(rng.choice(nI, n, replace=False)) for n in hl]
    hptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(hl, out=hptr[1:])
    hidx = np.concatenate(hist + [np.zeros(1)]).astype(np.int32)
    return U, I, user, pos, hptr, hidx


def _assert_same(got, want, what):
    for g, w, name in zip(got, want, ('ranks', 'targets', 'ids', 'values')):
        if g is None and w is None:
            continue
        bad = (g != w).reshape(g.shape[0], -1).any(1).nonzero().flatten()
        assert bad.numel() == 0, (what, name, bad[:8].tolist(), g[bad[:2]].tolist(), w[bad[:2]].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize('D', [64, 128, 256])
@pytest.mark.parametrize('R,nI', [(1, 10), (257, 300), (3000, 40_000), (90_000, 5_000)])
def test_exact_topk_lists_equal_the_fp32_path(D, R, nI, ws):
    U, I, user, pos, hptr, hidx = adversarial(D, R, nI, D + R)
    dU, dI, du, dp, dh, di = dv(U), dv(I), dv(user), dv(pos), dv(hptr), dv(hidx)
    for k in (1, 10, 20, 32):
        want = _lib.eval_rank_topk(dU, dI, du, dp, dh, di, ws, k=k, precision=0)[:4]
        got = _lib.eval_rank_topk(dU, dI, du, dp, dh, di, ws, k=k, precision=2)[:4]
        assert ws.status() == 0
        assert ws.last_topk_fallback_rows == 0
        _assert_same(got, want, f'k={k}')
        if R > 8 and nI > 3:                             # the user with three unmasked items: padded as precision 0 pads
            assert (got[2][8, 3:] == -1).all() and torch.isinf(got[3][8, 3:]).all()
        rs, tis, tvs = _lib.eval_rank_topk_shard(dU[du], dI, du, dp, U.shape[0], dh, di, want[1], ws, k=k, precision=2)
        assert ws.status() == 0
        _assert_same((rs, want[1], tis, tvs), want, f'item-shard entry point, k={k}')


@pytest.mark.gpu
def test_exact_topk_out_of_range_user_matches_the_fp32_path(ws):
    U, I, user, pos, hptr, hidx = adversarial(128, 257, 300, 5)
    user[20] = U.shape[0] + 3
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    want = _lib.eval_rank_topk(*args, ws, k=10, precision=0)
    st0 = ws.status()
    got = _lib.eval_rank_topk(*args, ws, k=10, precision=2)
    st2 = ws.status()
    assert st0 == st2 == 1
    ok = torch.from_numpy(user < U.shape[0]).to(DEV)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1][ok], want[1][ok])
    assert torch.equal(got[2], want[2]) and torch.equal(got[3], want[3])
    assert (got[2][20] == -1).all()


@pytest.mark.gpu
def test_exact_topk_overflowing_rows_are_rerun_alone(ws):
    """Rows whose scores rise with the item id put every item into the list; those rows, and only those, overflow their
    segment and are rerun at precision 0.  The lists still equal precision 0's."""
    rng = np.random.RandomState(2)
    D, R, nI, nU = 64, 600, 5000, 400
    I = (rng.randn(nI, D) * 0.5).astype(np.float32)
    I[:, 0] = np.arange(nI, dtype=np.float32) / nI * 4
    U = (rng.randn(nU, D) / 8).astype(np.float32)
    U[:, 0] = 0.0
    rising = np.arange(0, nU, 37)
    U[rising] = 0.0
    U[rising, 0] = 1.0
    user = rng.randint(0, nU, R).astype(np.int64)
    pos = rng.randint(0, nI, R).astype(np.int64)
    hl = rng.randint(0, 30, nU)
    hptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(hl, out=hptr[1:])
    hidx = np.concatenate([np.sort(rng.choice(nI, n, replace=False)) for n in hl] + [np.zeros(1)]).astype(np.int32)
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    n_rising = int(np.isin(user, rising).sum())
    assert n_rising > 0
    for k in (10, 32):
        want = _lib.eval_rank_topk(*args, ws, k=k, precision=0)[:4]
        got = _lib.eval_rank_topk(*args, ws, k=k, precision=2)[:4]
        assert ws.last_topk_fallback_rows == n_rising
        _assert_same(got, want, f'k={k}')
        rs, tis, tvs = _lib.eval_rank_topk_shard(args[0][args[2]], args[1], args[2], args[3], nU, args[4], args[5],
                                                 want[1], ws, k=k, precision=2)
        assert ws.last_topk_fallback_rows == n_rising
        _assert_same((rs, want[1], tis, tvs), want, f'item-shard, k={k}')


@pytest.mark.gpu
@pytest.mark.parametrize('G', [2, 3])
def test_exact_topk_on_emulated_item_shards(G, ws):
    """Item shards I[g::G] on one GPU: each shard's precision-2 lists, mapped to global ids and merged, equal the
    unsharded precision-0 lists; the per-shard counts add up to the ranks."""
    from whisprrec_b200 import sharded as S
    D, R, nI = 128, 3000, 20_000
    U, I, user, pos, hptr, hidx = adversarial(D, R, nI, 40 + G)
    du, dp = dv(user), dv(pos)
    for k in (10, 32):
        want = _lib.eval_rank_topk(dv(U), dv(I), du, dp, dv(hptr), dv(hidx), ws, k=k, precision=0)
        target = want[1]
        counts = torch.zeros(R, dtype=torch.int32, device=DEV)
        vs, ids = [], []
        for g in range(G):
            lay = S.ShardLayout(U.shape[0], nI, G, g)
            lp, li = lay.localise_history(hptr, hidx)
            rank_l, tki, tkv = _lib.eval_rank_topk_shard(dv(U[user]), dv(I[g::G]), du, lay.item_local_index(dp),
                                                         U.shape[0], dv(lp), dv(li), target, ws, k=k, precision=2)
            assert ws.status() == 0
            counts += rank_l - 1
            ids.append(lay.item_global_index(tki))
            vs.append(tkv)
        mv, mi = _lib.topk_merge(torch.stack(vs).contiguous(), torch.stack(ids).contiguous(), k)
        assert torch.equal(counts + 1, want[0])
        assert torch.equal(mi, want[2]) and torch.equal(mv, want[3])


@pytest.mark.gpu
@pytest.mark.parametrize('model_name', ['BPRMF', 'LightGCN', 'SGL'])
@pytest.mark.parametrize('D', [64, 256])
def test_ml100k_lists_at_precision_2_equal_precision_0(model_name, D):
    """Two seeded ml-100k epochs through BaseRunner, then rank_topk(dev, k=20) and recommend(dev, 20) at the default
    precision 2 against the same calls at precision 0."""
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.BPRMF import BPRMF
    from whisprrec_b200.models.general.LightGCN import LightGCN
    from whisprrec_b200.models.general.SGL import SGL
    from whisprrec_b200.utils import utils
    cls = {'BPRMF': BPRMF, 'LightGCN': LightGCN, 'SGL': SGL}[model_name]
    corpus = ml100k_corpus()
    args = model_args(cls, embedding_size=D)
    utils.init_seed(3407)
    model = cls(args, corpus).to(DEV)
    model.fuse()
    runner = BaseRunner(args)
    model.optimizer = runner._build_optimizer(model)
    data = {ph: cls.Dataset(model, corpus, ph) for ph in ('train', 'dev')}
    for _ in range(2):
        runner.fit(data['train'], epoch=1)
    # LightGCN and SGL propagate on every eval_tables() call, and the SpMM merges the slices of long rows with float
    # REDs, so two calls can differ in the last bits: both precisions score one propagation
    tables = tuple(t.clone() for t in model.eval_tables())
    model.eval_tables = lambda: tables
    assert runner.eval_precision == 2
    ws = model.tables.ws
    got = runner.rank_topk(data['dev'], k=20)[:4]
    items2, scores2 = runner.recommend(data['dev'], 20)
    assert ws.status() == 0 and ws.last_topk_fallback_rows == 0
    runner.eval_precision = 0
    want = runner.rank_topk(data['dev'], k=20)[:4]
    items0, scores0 = runner.recommend(data['dev'], 20)
    _assert_same(got, want, model_name)
    n = len(data['dev'])
    assert items2.shape == (n, 20) and items2.dtype == np.int64 and scores2.dtype == np.float32
    assert np.array_equal(items2, items0) and np.array_equal(scores2, scores0)
    assert np.array_equal(items0, want[2].cpu().numpy().astype(np.int64))
    items_default, _ = runner.recommend(data['dev'])
    assert items_default.shape == (n, max(runner.topk))
    # no history item is recommended
    hp, hi = corpus.history_csr()
    for r in range(0, n, 97):
        u = data['dev'].data['user_id'][r]
        assert not np.isin(items2[r], hi[hp[u]:hp[u + 1]]).any()
