"""Top-k lists of up to 256 items (wr_eval_rank_topk_long): precision 0's lists at precisions 0 and 2, one GPU and
item-sharded.  CPU: argument errors, the scratch query, the support predicate and a NumPy model of the range bound.
GPU: precision 0 against a NumPy FMA-chain oracle, precision 2 against precision 0 on adversarial tables, ranks against
k = 0 calls, the device-side row sweep, emulated item shards and ml-100k models through BaseRunner."""
import numpy as np
import pytest
import torch

from tests.helpers import ml100k_corpus, model_args
from whisprrec_b200 import _lib

DEV = torch.device('cuda:0')
KS = (33, 64, 100, 256)


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------

def test_long_topk_argument_errors_need_no_gpu():
    lib = _lib.load()
    # wr_eval_rank_topk_long(U, I, user, pos, R, n_users, n_items, D, hist_ptr, hist_idx, k, precision, topk_idx,
    #                        topk_val, rank, target, scratch, ws, stream)
    call = lambda D, k, p, tk=16, scratch=1024: lib.wr_eval_rank_topk_long(
        16, 16, 16, 16, 4, 4, 4, D, 16, 16, k, p, tk, tk, 16, 16, scratch, 16, None)
    # wr_eval_rank_topk_long_shard(Urows, I, user, pos_local, R, n_users, n_items, D, hist_ptr, hist_idx, k, precision,
    #                              target, topk_idx, topk_val, rank, scratch, ws, stream)
    shard = lambda D, k, p, tk=16, scratch=1024: lib.wr_eval_rank_topk_long_shard(
        16, 16, 16, 16, 4, 4, 4, D, 16, 16, k, p, 16, tk, tk, 16, scratch, 16, None)
    for f in (call, shard):
        for p in (0, 2):
            assert f(64, 0, p) == -4 and f(64, 257, p) == -4 and f(64, -1, p) == -4
            assert f(64, 100, p, scratch=None) == -1
            assert f(64, 100, p, tk=None) == -1                 # the lists are the point of the call
        assert f(64, 100, 1) == -4 and f(64, 33, 3) == -4      # precision 1 (approximate lists) is refused
        assert f(32, 100, 2) == -3 and f(16, 100, 2) == -3 and f(512, 100, 2) == -3
        assert f(512, 100, 0) == -3 and f(12, 100, 0) == -3
    assert lib.wr_eval_rank_topk_long(16, 16, 16, 16, 4, 4, 4, 64, 16, 16, 100, 2, 16, None, 16, 16, 1024, 16,
                                      None) == -1              # one of the two list outputs missing
    assert lib.wr_eval_rank_topk_long_shard(16, 16, 16, 16, 4, 4, 4, 64, 16, 16, 100, 0, None, 16, 16, 16, 1024, 16,
                                            None) == -1        # no target scores
    # wr_topk_merge_long(val, idx, world, R, k, out_val, out_idx, stream)
    assert lib.wr_topk_merge_long(16, 16, 2, 4, 0, 16, 16, None) == -4
    assert lib.wr_topk_merge_long(16, 16, 2, 4, 257, 16, 16, None) == -4
    assert lib.wr_topk_merge_long(None, 16, 2, 4, 100, 16, 16, None) == -1
    assert lib.wr_topk_merge_long(16, 16, 0, 4, 100, 16, 16, None) == -2
    # the k <= 32 contract is unchanged
    assert lib.wr_topk_merge(16, 16, 2, 4, 33, 16, 16, None) == -4


def test_long_topk_scratch_query():
    lib = _lib.load()
    q = lib.wr_eval_scratch_bytes_topk_long
    per_row = 16 * 4 + 4 + 4096 * 4
    for R, n in ((1, 10), (3000, 40_000), (90_000, 5_000), (262_144, 1_000_000), (1_000_000, 1_000)):
        for D in (64, 128, 256):
            for p in (0, 2):
                sizes = [q(R, n, D, p, k) for k in (1, 32, 33, 64, 100, 256)]
                assert all(s > 0 for s in sizes) and sizes == sorted(sizes)       # never shrinks with k
                rows = min(R, 65_536) if p == 0 else None
                base = 1024 + (lib.wr_eval_scratch_bytes(R, n, D, 2) if p == 2 else 0)
                tail = sizes[-1] - base
                # one row block's bounds, counts and 4,096-id segments: at most 65,536 rows, so <= 1 GB of segments
                assert tail <= 65_536 * per_row + 3 * 1024
                assert tail >= min(R, 256) * per_row
                if rows is not None:
                    assert rows * per_row <= tail <= rows * per_row + 3 * 1024
            assert q(2 * R, n, D, 0, 100) >= q(R, n, D, 0, 100)                    # grows with the rows
            assert q(2 * R, n, D, 2, 100) >= q(R, n, D, 2, 100)
    assert q(3000, 5000, 64, 0, 100) > q(1000, 5000, 64, 0, 100)
    assert q(3000, 5000, 64, 2, 100) > q(1000, 5000, 64, 2, 100)
    assert q(1000, 5000, 32, 0, 100) > 0 and q(1000, 5000, 32, 2, 100) == 0
    for k in (0, 257):
        assert q(1000, 5000, 64, 0, k) == 0 and q(1000, 5000, 64, 2, k) == 0
    assert q(1000, 5000, 64, 1, 100) == 0
    # the k <= 32 query is unchanged
    assert lib.wr_eval_scratch_bytes_topk(1000, 5000, 64, 0, 10) == 0


def test_long_topk_support_truth_table():
    for D in (16, 32, 64, 128, 256, 512):
        for k in (0, 1, 10, 32, 33, 64, 100, 256, 257):
            assert _lib.exact_tc_topk_long_supported(D, k) == (D in (64, 128, 256) and 1 <= k <= 256), (D, k)
            # the k <= 32 predicate is unchanged
            assert _lib.exact_tc_topk_supported(D, k) == (D in (64, 128, 256) and 1 <= k <= 32), (D, k)
    assert not _lib.exact_tc_topk_supported(128, 33)


def _floor(L, eps):
    """exact_topk_floor in fp32: L - (2 eps + 2.4e-7 |L|)."""
    L = np.float32(L)
    return np.float32(L - np.float32(np.float32(2 * eps) + np.float32(2.4e-7) * np.float32(abs(L))))


def _range_bound(x, k, tile):
    """The bound pass on one row: S = ceil(k / 32) or more ranges of whole tiles (the last may be short), the k'-th best
    of each (k' = ceil(k / S), -inf if the range has fewer), and the S-th largest of those."""
    n_tiles = -(-len(x) // tile)
    s = -(-k // 32)
    kp = -(-k // s)
    assert kp <= 32 and s * kp >= k
    if n_tiles < s:
        return -np.inf
    tpr = n_tiles // s
    bounds = []
    for c in range(-(-n_tiles // tpr)):
        v = np.sort(x[c * tpr * tile:(c + 1) * tpr * tile])[::-1]
        v = v[np.isfinite(v)]
        bounds.append(v[kp - 1] if len(v) >= kp else -np.inf)
    return sorted(bounds)[::-1][s - 1]


@pytest.mark.parametrize('kind', ['random', 'adversarial', 'tied'])
def test_long_topk_range_bound_keeps_the_exact_lists(kind):
    """The rule of both precisions on modelled scores: s exact, t = s + noise with |t - s| <= eps / 2 (eps as the kernel
    passes it).  L over s is <= the k-th best s; L over t, lowered by 2 eps, keeps every item of the exact top k; the
    candidates sorted by (s desc, id asc) give the exact list."""
    rng = np.random.RandomState({'random': 1, 'adversarial': 2, 'tied': 3}[kind])
    n = 9030                                             # a short last tile
    for trial in range(4):
        if kind == 'random':
            s = rng.randn(n).astype(np.float32)
        elif kind == 'adversarial':                          # rising with the id, one hot range, a flat plateau
            s = np.linspace(-1, 1, n).astype(np.float32) if trial % 2 == 0 else rng.randn(n).astype(np.float32)
            s[2000:2300] += np.float32(5)
            s[5000:7000] = np.float32(0.5)
        else:
            s = np.round(rng.randn(n) * 3).astype(np.float32) / np.float32(4)
        s[rng.choice(n, 60, replace=False)] = -np.inf        # history
        eps = np.float32(1e-3 * (trial + 1))
        t = (s + rng.uniform(-0.5, 0.5, n).astype(np.float32) * eps).astype(np.float32)
        t[~np.isfinite(s)] = -np.inf
        finite = np.flatnonzero(np.isfinite(s))
        order = finite[np.lexsort((finite, -s[finite]))]
        for k in KS:
            want = order[:k]
            sk = s[want[-1]]
            for tile in (64, 256):
                Ls = _range_bound(s, k, tile)
                assert np.isfinite(Ls) and Ls <= sk, (k, tile)
                cand = np.flatnonzero(np.isfinite(s) & (s >= Ls))
                assert set(want) <= set(cand)
                got = cand[np.lexsort((cand, -s[cand]))][:k]
                assert np.array_equal(got, want)
                Lt = _range_bound(t, k, tile)
                cand = np.flatnonzero(np.isfinite(t) & (t >= _floor(Lt, eps)))
                assert set(want) <= set(cand), (kind, trial, k, tile)
                got = cand[np.lexsort((cand, -s[cand]))][:k]
                assert np.array_equal(got, want)


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


def _fma_chain_oracle(A, B):
    """precision 0's scores [len(A), len(B)]: s = fmaf(a_d, b_d, s), d = 0 .. D-1, with fmaf's single rounding: the
    product is exact in float64, the sum's float64 rounding error is recovered (TwoSum) and folded in by rounding to odd,
    so the one rounding to float32 is the correct one."""
    s = np.zeros((A.shape[0], B.shape[0]), dtype=np.float32)
    for d in range(A.shape[1]):
        x = A[:, d, None].astype(np.float64) * B[None, :, d].astype(np.float64)
        y = s.astype(np.float64)
        z = x + y
        bp = z - x
        err = (x - (z - bp)) + (y - bp)
        even = (z.view(np.int64) & 1) == 0
        z = np.where((err != 0) & even, np.nextafter(z, np.where(err > 0, np.inf, -np.inf)), z)
        s = z.astype(np.float32)
    return s


def _oracle_lists(U, I, user, pos, hptr, hidx, k, shard=False):
    """(ids, values) of every row: unmasked items by (value desc, id asc), padded with (-1, -inf)."""
    R = len(user)
    ids = np.full((R, k), -1, dtype=np.int32)
    vals = np.full((R, k), -np.inf, dtype=np.float32)
    ok = (user >= 0) & (user < U.shape[0])
    if not shard:
        ok &= (pos >= 0) & (pos < I.shape[0])
    rows = np.flatnonzero(ok)
    S = _fma_chain_oracle(U[user[rows]], I)
    for q, r in enumerate(rows):
        u = user[r]
        s = S[q].copy()
        s[hidx[hptr[u]:hptr[u + 1]]] = -np.inf
        cand = np.flatnonzero(s > -np.inf)
        top = cand[np.lexsort((cand, -s[cand]))][:k]
        ids[r, :len(top)] = top
        vals[r, :len(top)] = s[top]
    return ids, vals


def tables(D, R, nI, seed, nU=400):
    """Random tables with a user whose history leaves three items (fewer than k) and an all-zero user (every score 0:
    the list is the first items by id)."""
    rng = np.random.RandomState(seed)
    U = (rng.randn(nU, D) / np.sqrt(D)).astype(np.float32)
    I = (rng.randn(nI, D) * rng.uniform(0.5, 1.5, (nI, 1))).astype(np.float32)
    U[11] = 0.0
    user = rng.randint(0, nU, R).astype(np.int64)
    user[:min(R, 3)] = 11
    if R > 8:
        user[8] = 12
    pos = rng.randint(0, nI, R).astype(np.int64)
    hl = rng.randint(0, min(50, nI), nU)
    hl[12] = max(0, nI - 3)
    hist = [np.sort(rng.choice(nI, n, replace=False)) for n in hl]
    hptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(hl, out=hptr[1:])
    hidx = np.concatenate(hist + [np.zeros(1)]).astype(np.int32)
    return U, I, user, pos, hptr, hidx


def _tied_rows(user, hptr, nI):
    """Rows of the all-zero user 11 (every score 0: all items tie) whose unmasked items overflow a 4,096-id segment: the
    row sweep finishes them."""
    return int((user == 11).sum()) if nI - (hptr[12] - hptr[11]) > 4096 else 0


def _assert_same(got, want, what):
    for g, w, name in zip(got, want, ('ranks', 'targets', 'ids', 'values')):
        bad = (g != w).reshape(g.shape[0], -1).any(1).nonzero().flatten()
        assert bad.numel() == 0, (what, name, bad[:8].tolist(), g[bad[:2]].tolist(), w[bad[:2]].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize('D', [16, 64, 256])
@pytest.mark.parametrize('R,nI', [(1, 10), (300, 200), (257, 5000)])
def test_long_lists_at_precision_0_equal_the_numpy_oracle(D, R, nI, ws):
    """Bit-identical ids and values, including rows padded because n_items < k or the history leaves fewer than k."""
    U, I, user, pos, hptr, hidx = tables(D, R, nI, D + R)
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    for k in KS:
        rank, target, ids, vals, _ = _lib.eval_rank_topk(*args, ws, k=k, precision=0)
        assert ws.last_topk_fallback_rows == _tied_rows(user, hptr, nI)
        wi, wv = _oracle_lists(U, I, user, pos, hptr, hidx, k)
        assert np.array_equal(ids.cpu().numpy(), wi), k
        assert np.array_equal(vals.cpu().numpy().view(np.int32), wv.view(np.int32)), k
        if R > 8:
            assert (ids[8, 3:] == -1).all() and torch.isinf(vals[8, 3:]).all()
        if nI < k:
            assert (ids[:, nI:] == -1).all()


@pytest.mark.gpu
def test_long_lists_out_of_range_user(ws):
    U, I, user, pos, hptr, hidx = tables(64, 257, 3000, 5)
    user[20] = U.shape[0] + 3
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    for p in (0, 2):
        rank, target, ids, vals, _ = _lib.eval_rank_topk(*args, ws, k=100, precision=p)
        assert ws.status() == 1                              # WR_STATUS_INDEX_OUT_OF_RANGE, as the k <= 32 lists raise
        wi, wv = _oracle_lists(U, I, user, pos, hptr, hidx, 100)
        assert np.array_equal(ids.cpu().numpy(), wi) and np.array_equal(vals.cpu().numpy(), wv)
        assert (ids[20] == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize('D', [32, 128])
def test_long_path_at_short_k_equals_the_k32_lists(D, ws):
    """The long entry point at k in {1, 10, 32} returns what wr_eval_rank_topk returns at precision 0."""
    U, I, user, pos, hptr, hidx = tables(D, 700, 6000, 7)
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    for k in (1, 10, 32):
        want = _lib.eval_rank_topk(*args, ws, k=k, precision=0)[:4]
        for p in ((0, 2) if D == 128 else (0,)):
            got = _lib._eval_rank_topk_long(*args, ws, k, p)[:4]
            _assert_same(got, want, f'k={k} precision {p}')


@pytest.mark.gpu
@pytest.mark.parametrize('D', [64, 128, 256])
@pytest.mark.parametrize('R,nI', [(1, 10), (257, 300), (3000, 40_000), (90_000, 5_000)])
def test_long_lists_at_precision_2_equal_precision_0(D, R, nI, ws):
    """Adversarial tables (duplicated items, an all-zero user, long histories, a user with three unmasked items): ids,
    values and order equal precision 0's; ranks and targets equal the k = 0 calls at each precision."""
    from tests.test_eval_topk_exact import adversarial
    U, I, user, pos, hptr, hidx = adversarial(D, R, nI, D + R + 1)
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    ranks = {p: _lib.eval_rank_topk(*args, ws, k=0, precision=p)[:2] for p in (0, 2)}
    for k in KS:
        want = _lib.eval_rank_topk(*args, ws, k=k, precision=0)[:4]
        got = _lib.eval_rank_topk(*args, ws, k=k, precision=2)[:4]
        assert ws.status() == 0 and ws.last_topk_fallback_rows == _tied_rows(user, hptr, nI)
        _assert_same(got, want, f'k={k}')
        _assert_same(want[:2], ranks[0], f'precision 0 ranks, k={k}')
        _assert_same(got[:2], ranks[2], f'precision 2 ranks, k={k}')
        rs, tis, tvs = _lib.eval_rank_topk_shard(args[0][args[2]], args[1], args[2], args[3], U.shape[0], args[4],
                                                 args[5], want[1], ws, k=k, precision=2)
        assert ws.status() == 0
        _assert_same((rs, want[1], tis, tvs), want, f'item-shard entry point, k={k}')


@pytest.mark.gpu
@pytest.mark.parametrize('table', ['equal', 'rising'])
def test_long_lists_overflowing_rows_are_swept_on_the_device(table, ws):
    """All-equal item rows (every item ties) and scores rising with the item id put most items above the bound: those
    rows overflow their 4,096-id segment and the row sweep finishes them.  The lists equal the oracle at both
    precisions."""
    rng = np.random.RandomState(4)
    D, R, nI, nU = 64, 40, 12_000, 50
    U = (rng.randn(nU, D) / 8).astype(np.float32)
    if table == 'equal':
        I = np.repeat((rng.randn(1, D) * 0.5).astype(np.float32), nI, 0)
    else:
        I = (rng.randn(nI, D) * 0.01).astype(np.float32)
        I[:, 0] = np.arange(nI, dtype=np.float32) / nI * 4
        U[:, 0] = 1.0
        U[:, 1:] = 0.0
    user = rng.randint(0, nU, R).astype(np.int64)
    pos = rng.randint(0, nI, R).astype(np.int64)
    hl = rng.randint(0, 30, nU)
    hptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(hl, out=hptr[1:])
    hidx = np.concatenate([np.sort(rng.choice(nI, n, replace=False)) for n in hl] + [np.zeros(1)]).astype(np.int32)
    args = [dv(x) for x in (U, I, user, pos, hptr, hidx)]
    ranks = {p: _lib.eval_rank_topk(*args, ws, k=0, precision=p)[:2] for p in (0, 2)}
    for k in (64, 256):
        wi, wv = _oracle_lists(U, I, user, pos, hptr, hidx, k)
        for p in (0, 2):
            rank, target, ids, vals, _ = _lib.eval_rank_topk(*args, ws, k=k, precision=p)
            # rising scores: a short last range of high scores can lift the bound enough at k = 64 (precision 2's
            # 256-item tiles); at k = 256 the bound is the 8th largest of 9-10 ranges and every row overflows
            if table == 'equal' or k == 256:
                assert ws.last_topk_fallback_rows > 0, (p, k)
            assert np.array_equal(ids.cpu().numpy(), wi), (p, k)
            assert np.array_equal(vals.cpu().numpy(), wv), (p, k)
            _assert_same((rank, target), ranks[p], f'ranks, precision {p}')


@pytest.mark.gpu
@pytest.mark.parametrize('G', [2, 3])
def test_long_lists_on_emulated_item_shards(G, ws):
    """Item shards I[g::G] on one GPU: each shard's long lists, mapped to global ids and merged, equal the unsharded
    precision-0 lists; the per-shard counts add up to the ranks."""
    from tests.test_eval_topk_exact import adversarial
    from whisprrec_b200 import sharded as S
    D, R, nI = 128, 3000, 20_000
    U, I, user, pos, hptr, hidx = adversarial(D, R, nI, 50 + G)
    du, dp = dv(user), dv(pos)
    for k in (64, 256):
        want = _lib.eval_rank_topk(dv(U), dv(I), du, dp, dv(hptr), dv(hidx), ws, k=k, precision=0)
        for p in (2, 0):
            counts = torch.zeros(R, dtype=torch.int32, device=DEV)
            vs, ids = [], []
            for g in range(G):
                lay = S.ShardLayout(U.shape[0], nI, G, g)
                lp, li = lay.localise_history(hptr, hidx)
                rank_l, tki, tkv = _lib.eval_rank_topk_shard(dv(U[user]), dv(I[g::G]), du, lay.item_local_index(dp),
                                                             U.shape[0], dv(lp), dv(li), want[1], ws, k=k, precision=p)
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
def test_ml100k_recommend_100_at_precision_2_equals_precision_0(model_name, D):
    """Two seeded ml-100k epochs with --topk 10,50,100, then recommend(dev) (k = 100 by default) at precision 2 against
    precision 0; k = 257 is refused before any GPU work."""
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.BPRMF import BPRMF
    from whisprrec_b200.models.general.LightGCN import LightGCN
    from whisprrec_b200.models.general.SGL import SGL
    from whisprrec_b200.utils import utils
    cls = {'BPRMF': BPRMF, 'LightGCN': LightGCN, 'SGL': SGL}[model_name]
    corpus = ml100k_corpus()
    args = model_args(cls, embedding_size=D, topk='10,50,100')
    utils.init_seed(3407)
    model = cls(args, corpus).to(DEV)
    model.fuse()
    runner = BaseRunner(args)
    model.optimizer = runner._build_optimizer(model)
    data = {ph: cls.Dataset(model, corpus, ph) for ph in ('train', 'dev')}
    for _ in range(2):
        runner.fit(data['train'], epoch=1)
    # both precisions score one propagation (LightGCN and SGL re-propagate with float REDs on every call)
    tables = tuple(t.clone() for t in model.eval_tables())
    model.eval_tables = lambda: tables
    assert runner.eval_precision == 2
    ws = model.tables.ws
    items2, scores2 = runner.recommend(data['dev'])
    assert ws.status() == 0 and ws.last_topk_fallback_rows == 0
    with pytest.raises(ValueError, match='256'):
        runner.recommend(data['dev'], 257)
    runner.eval_precision = 0
    items0, scores0 = runner.recommend(data['dev'])
    n = len(data['dev'])
    assert items2.shape == (n, 100) and items2.dtype == np.int64 and scores2.dtype == np.float32
    assert np.array_equal(items2, items0) and np.array_equal(scores2, scores0)
    assert (items2[:, :20] >= 0).all()
    hp, hi = corpus.history_csr()
    for r in range(0, n, 97):
        u = data['dev'].data['user_id'][r]
        assert not np.isin(items2[r], hi[hp[u]:hp[u + 1]]).any()
    # the first 10 entries are the k = 10 list
    runner.eval_precision = 2
    items10, _ = runner.recommend(data['dev'], 10)
    assert np.array_equal(items10, items2[:, :10])
