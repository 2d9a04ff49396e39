#!/usr/bin/env python
"""Worker for the multi-rank tests; launched by tests/test_multi_gpu.py (and by hand on a GPU box):

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tests/dist_worker.py gpu
    torchrun ... tests/dist_worker.py cpu         # gloo: the host-side shard logic with the oracle as the compute

`gpu`: one B200 per rank.  The sharded BPRMF step, LightGCN step and item-sharded evaluation must reproduce the
single-GPU kernels run by the same rank on the whole batch / whole tables (SURVEY.md section 8e: "G in {2,4,8}
results equal G = 1").  The per-rank body, check_sharded_paths, also runs on one GPU with emulated ranks in threads
(tests/test_sharded_emulated.py).
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.helpers import assert_close  # noqa: E402
from whisprrec_b200.sharded import ShardLayout, combine_shard_ranks  # noqa: E402


def problem(seed, nU, nI, D, n_pairs):
    rng = np.random.RandomState(seed)
    U = (rng.randn(nU, D) * 0.1).astype(np.float32)
    I = (rng.randn(nI, D) * 0.1).astype(np.float32)
    pairs = np.unique(np.stack([rng.randint(0, nU, n_pairs), rng.randint(0, nI, n_pairs)], 1), axis=0)
    return rng, U, I, pairs


# --------------------------------------------------------------------------------------------------------------
# gloo / CPU: host logic only, the oracle computes
# --------------------------------------------------------------------------------------------------------------
def run_cpu():
    from oracle import whispr_oracle as O
    dist.init_process_group('gloo')
    rank, world = dist.get_rank(), dist.get_world_size()
    nU, nI, D = 37, 53, 16
    rng, U, I, pairs = problem(11, nU, nI, D, 600)
    lay = ShardLayout(nU, nI, world, rank)

    # every row has exactly one owner and the shards tile the tables
    full = np.concatenate([U, I])
    shard = lay.shard_of_table(full)
    nodes = lay.local_nodes()
    assert (shard[nodes >= 0] == full[nodes[nodes >= 0]]).all() and (shard[nodes < 0] == 0).all()
    owned = torch.zeros(nU + nI, dtype=torch.int64)
    owned[torch.from_numpy(nodes[nodes >= 0])] = 1
    dist.all_reduce(owned)
    assert (owned == 1).all()

    # batch slices tile the batch
    B = 101
    lo, hi = lay.batch_slice(B)
    cover = torch.zeros(B, dtype=torch.int64)
    cover[lo:hi] = 1
    dist.all_reduce(cover)
    assert (cover == 1).all()

    # data-parallel step == single-process step: per-rank gradient of its slice (scaled by the GLOBAL batch) summed
    sel = rng.randint(0, len(pairs), B)
    user, pos, neg = pairs[sel, 0], pairs[sel, 1], rng.randint(1, nI, B)
    loss_full, gU_full, gI_full = O.bpr_fwd_bwd(U, I, user, pos, neg)
    l, gU, gI = O.bpr_fwd_bwd(U, I, user[lo:hi], pos[lo:hi], neg[lo:hi])
    scale = (hi - lo) / B
    part = torch.cat([gU.reshape(-1) * scale, gI.reshape(-1) * scale, torch.tensor([float(l) * scale])])
    dist.all_reduce(part)
    assert_close(part[:-1].numpy(), torch.cat([gU_full.reshape(-1), gI_full.reshape(-1)]).numpy(), 'sharded grads')
    assert abs(float(part[-1]) - float(loss_full)) < 1e-6

    # item-sharded evaluation: local counts + local top-k, combined, equal the unsharded oracle
    hp, hi_ = O.history_csr(nU, pairs[: len(pairs) // 2], pairs[:1])
    eu, ep = pairs[len(pairs) // 2:, 0].astype(np.int64), pairs[len(pairs) // 2:, 1].astype(np.int64)
    S = O.full_scores(U, I, eu).numpy()
    want_rank, target = O.ranks_count(S, eu, ep, hp, hi_)
    k = 5
    want_topk = O.topk_masked(S, eu, hp, hi_, k)[0]
    lptr, lidx = lay.localise_history(hp, hi_)
    mine = lay.local_items()
    S_local = S[:, mine]
    cnt = np.zeros(len(eu), dtype=np.int64)
    cand_v = np.full((len(eu), k), -np.inf, dtype=np.float32)
    cand_i = np.full((len(eu), k), -1, dtype=np.int64)
    for r, u in enumerate(eu):
        s = S_local[r].copy()
        s[lidx[lptr[u]:lptr[u + 1]]] = -np.inf
        cnt[r] = 1 + np.count_nonzero(s > target[r])
        order = np.lexsort((np.arange(len(s)), -s))[:k]
        order = order[np.isfinite(s[order])]
        cand_v[r, :len(order)] = s[order]
        cand_i[r, :len(order)] = lay.item_global_index(order)
    pl = lay.item_local_index(ep)
    assert ((pl >= 0) == (ep % world == rank)).all() and (mine[pl[pl >= 0]] == ep[pl >= 0]).all()
    gathered = [torch.zeros(len(eu), dtype=torch.int64) for _ in range(world)]
    dist.all_gather(gathered, torch.from_numpy(cnt))
    got_rank = combine_shard_ranks(gathered).numpy()
    assert (got_rank == want_rank).all()
    gv = [torch.zeros((len(eu), k)) for _ in range(world)]
    gi = [torch.zeros((len(eu), k), dtype=torch.int64) for _ in range(world)]
    dist.all_gather(gv, torch.from_numpy(cand_v))
    dist.all_gather(gi, torch.from_numpy(cand_i))
    av, ai = torch.cat(gv, 1).numpy(), torch.cat(gi, 1).numpy()
    for r in range(len(eu)):
        order = np.lexsort((ai[r], -av[r]))[:k]
        got = ai[r][order]
        assert (got[got >= 0] == want_topk[r][:len(got[got >= 0])]).all()

    # LightGCN row partition: local rows of the adjacency, propagated with all-gathered inputs, tile the full product
    rowptr, col, val = O.build_norm_adj_csr(nU, nI, pairs[:, 0], pairs[:, 1])
    lptr2, lcol, src = lay.local_adjacency(rowptr, col)
    A_full = O.csr_to_torch(rowptr, col, val, nU + nI)
    Y_full = torch.sparse.mm(A_full, torch.from_numpy(full)).numpy()
    A_loc = O.csr_to_torch(lptr2, lcol, val[src], nU + nI) if len(lcol) else None
    A_loc = torch.sparse_csr_tensor(torch.from_numpy(lptr2), torch.from_numpy(lcol.astype(np.int64)),
                                    torch.from_numpy(val[src]), size=(lay.n_local, nU + nI))
    Y_loc = torch.sparse.mm(A_loc, torch.from_numpy(full)).numpy()
    assert_close(Y_loc[nodes >= 0], Y_full[nodes[nodes >= 0]], 'row-partitioned SpMM')
    assert (Y_loc[nodes < 0] == 0).all()
    dist.barrier()
    if rank == 0:
        print('dist_worker cpu ok: world', world)
    dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------------------
# NCCL / one B200 per rank
# --------------------------------------------------------------------------------------------------------------
def run_gpu():
    from whisprrec_b200 import sharded as S
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    assert torch.cuda.device_count() >= dist.get_world_size(), \
        'one GPU per rank (never share a GPU between spinning ranks)'
    peers = S.PeerGroup(dev)
    check_sharded_paths(peers)
    peers.close()
    dist.destroy_process_group()


def check_sharded_paths(peers):
    """The per-rank body of the `gpu` mode on one rank of `peers` (a PeerGroup, or anything with its interface: world,
    rank, device, ws, dist, group, alloc, alloc_bytes, host_sync, barrier).  Prints five `dist_worker gpu ok` lines on
    rank 0."""
    from oracle import whispr_oracle as O
    from whisprrec_b200 import _lib
    from whisprrec_b200 import sharded as S
    rank, world, dev = peers.rank, peers.world, peers.device
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    host = lambda t: t.detach().cpu().numpy()

    for (nU, nI, D, B) in [(301, 517, 64, 2048), (64, 40, 16, 333), (1000, 3000, 128, 4096)]:
        rng, U, I, pairs = problem(5, nU, nI, D, 20 * nU)
        lay = S.ShardLayout(nU, nI, world, rank)
        # ---------------- BPRMF: three sharded steps against the single-GPU step on the whole batch ----------------
        tabs = S.ShardedTables(peers, lay, D)
        tabs.load_full(d(U), d(I))
        Pf = d(np.concatenate([U, I]))
        Mf, Vf, Gf = torch.zeros_like(Pf), torch.zeros_like(Pf), torch.zeros_like(Pf)
        ws, lossf = _lib.Workspace(dev), torch.zeros(1, device=dev)
        for step in range(1, 4):
            sel = rng.randint(0, len(pairs), B)
            user, pos, neg = pairs[sel, 0].astype(np.int64), pairs[sel, 1].astype(np.int64), rng.randint(1, nI, B).astype(np.int64)
            lo, hi = lay.batch_slice(B)
            loss = S.bprmf_step(tabs, d(user[lo:hi]), d(pos[lo:hi]), d(neg[lo:hi]), B, 1e-3, 1e-6)
            loss_v = float(loss[0])
            _lib.bpr_fwd_bwd(Pf[:nU], Pf[nU:], d(user), d(pos), d(neg), Gf[:nU], Gf[nU:], lossf, ws)
            _lib.adam_l2_sweep(Pf, Mf, Vf, Gf, step, 1e-3, 1e-6)
            assert abs(loss_v - float(lossf[0])) <= 2e-6 * abs(float(lossf[0])), (loss_v, float(lossf[0]))
            gu, gi = tabs.gather_full()
            assert_close(host(gu), host(Pf[:nU]), f'sharded U step {step}', rtol=1e-5, atol_scale=2e-6)
            assert_close(host(gi), host(Pf[nU:]), f'sharded I step {step}', rtol=1e-5, atol_scale=2e-6)
            peers.barrier()
        assert float(tabs.G.abs().max()) == 0.0 and tabs.ws.status() == 0

        # ---------------- the multi-launch form with the staged (inbox) gradient scatter: large batches ----------------
        if D == 128:
            Bs = 8192 * world                               # 8,192 rows per rank: the staged protocol
            tabs3 = S.ShardedTables(peers, lay, D)
            tabs3.load_full(d(U), d(I))
            tabs3.single_launch = False                     # what shards too large for the cooperative step take
            Pf3 = d(np.concatenate([U, I]))
            Mf3, Vf3, Gf3 = torch.zeros_like(Pf3), torch.zeros_like(Pf3), torch.zeros_like(Pf3)
            for step in range(1, 4):
                sel = rng.randint(0, len(pairs), Bs)
                user, pos, neg = pairs[sel, 0].astype(np.int64), pairs[sel, 1].astype(np.int64), rng.randint(1, nI, Bs).astype(np.int64)
                lo, hi = lay.batch_slice(Bs)
                loss = S.bprmf_step(tabs3, d(user[lo:hi]), d(pos[lo:hi]), d(neg[lo:hi]), Bs, 1e-3, 1e-6)
                loss_v = float(loss[0])
                _lib.bpr_fwd_bwd(Pf3[:nU], Pf3[nU:], d(user), d(pos), d(neg), Gf3[:nU], Gf3[nU:], lossf, ws)
                _lib.adam_l2_sweep(Pf3, Mf3, Vf3, Gf3, step, 1e-3, 1e-6)
                assert abs(loss_v - float(lossf[0])) <= 2e-6 * abs(float(lossf[0])), (loss_v, float(lossf[0]))
                gu, gi = tabs3.gather_full()
                assert_close(host(gu), host(Pf3[:nU]), f'staged scatter U step {step}', rtol=1e-5, atol_scale=2e-6)
                assert_close(host(gi), host(Pf3[nU:]), f'staged scatter I step {step}', rtol=1e-5, atol_scale=2e-6)
                peers.barrier()
            assert getattr(tabs3, '_inbox', None) is not None and int(tabs3._inbox['idx'].abs().max()) == 0
            assert float(tabs3.G.abs().max()) == 0.0 and tabs3.ws.status() == 0

        # ---------------- evaluation: items sharded, ranks / top-k equal the single-GPU kernel ----------------
        half = len(pairs) // 2
        hp, hi_ = O.history_csr(nU, pairs[:half], pairs[:1])
        eu, ep = pairs[half:, 0].astype(np.int64), pairs[half:, 1].astype(np.int64)
        lh = lay.localise_history(hp, hi_)
        lh = (d(lh[0]), d(lh[1]))
        Uf, If = Pf[:nU].contiguous(), Pf[nU:].contiguous()
        want = _lib.eval_rank_topk(Uf, If, d(eu), d(ep), d(hp), d(hi_), ws, k=10)
        got = S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), d(eu), d(ep), lh, k=10)
        # parameters differ by the REDs' summation order (1e-6 relative), so compare through the sharded tables
        gu, gi = tabs.gather_full()
        want = _lib.eval_rank_topk(gu.contiguous(), gi.contiguous(), d(eu), d(ep), d(hp), d(hi_), ws, k=10)
        assert (host(got[0]) == host(want[0])).all(), 'sharded ranks'
        assert (host(got[1]) == host(want[1])).all(), 'sharded targets'
        assert (host(got[2]) == host(want[2])).all(), 'sharded top-k ids'
        assert (host(got[3]) == host(want[3])).all(), 'sharded top-k values'
        # lists longer than 32 items: the long-list kernels per shard and the long merge
        want = _lib.eval_rank_topk(gu.contiguous(), gi.contiguous(), d(eu), d(ep), d(hp), d(hi_), ws, k=100)
        got = S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), d(eu), d(ep), lh, k=100)
        for g_, w_, what in zip(got, want, ('ranks', 'targets', 'top-100 ids', 'top-100 values')):
            assert (host(g_) == host(w_)).all(), 'sharded ' + what
        if D in (64, 128):
            want_tc = _lib.eval_rank_topk(gu.contiguous(), gi.contiguous(), d(eu), d(ep), d(hp), d(hi_), ws, precision=1)
            got_tc = S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), d(eu), d(ep), lh, precision=1)
            assert (host(got_tc[1]) == host(want_tc[1])).all(), 'sharded tensor-core targets'
            assert np.mean(host(got_tc[0]) != host(want_tc[0])) < 2e-3, 'sharded tensor-core ranks'

        # ---------------- LightGCN: L = 2 sharded steps against the oracle on the whole batch ----------------
        # third pass: a batch of 8,192 rows per rank -> the row exchange (owners deliver the pooled rows, EmbLoss computed
        # by the owners of the ego rows from the request lists), with the fused all-gather of the layer outputs
        for gather_first, B in ((False, B), (True, B), (True, 8192 * world)):
            L, reg = 2, 1e-5
            rowptr, col, val = O.build_norm_adj_csr(nU, nI, pairs[:, 0], pairs[:, 1])
            dinv = O.deg_inv_sqrt(np.diff(rowptr))
            tabs2 = S.ShardedTables(peers, lay, D)
            tabs2.load_full(d(U), d(I))
            lg = S.ShardedLightGCN(tabs2, rowptr, col, dinv, L, reg, gather_first=gather_first)
            A = O.csr_to_torch(rowptr, col, val, nU + nI)
            oU, oI = torch.from_numpy(U.copy()), torch.from_numpy(I.copy())
            om = [torch.zeros_like(oU), torch.zeros_like(oU), torch.zeros_like(oI), torch.zeros_like(oI)]
            for step in range(1, 3):
                sel = rng.randint(0, len(pairs), B)
                user, pos, neg = pairs[sel, 0].astype(np.int64), pairs[sel, 1].astype(np.int64), rng.randint(1, nI, B).astype(np.int64)
                lo, hi = lay.batch_slice(B)
                loss = lg.step(d(user[lo:hi]), d(pos[lo:hi]), d(neg[lo:hi]), B, 1e-3, 0.0)
                o_loss, ogU, ogI = O.lightgcn_fwd_bwd(A, oU, oI, user, pos, neg, L, reg)
                O.adam_l2_step(oU, om[0], om[1], ogU, step, 1e-3, 0.0)
                O.adam_l2_step(oI, om[2], om[3], ogI, step, 1e-3, 0.0)
                assert abs(float(loss[0]) - float(o_loss)) <= 1e-5 * abs(float(o_loss)), (float(loss[0]), float(o_loss))
                gu, gi = tabs2.gather_full()
                assert_close(host(gu), oU.numpy(), f'sharded LightGCN U step {step}', rtol=1e-4, atol_scale=1e-4)
                assert_close(host(gi), oI.numpy(), f'sharded LightGCN I step {step}', rtol=1e-4, atol_scale=1e-4)
                peers.barrier()
            lg.propagate()
            pu, pi = tabs2.gather_full(lg.pool_T)
            o_pool = O.lightgcn_propagate(A, torch.cat([oU, oI]), L).numpy()
            assert_close(host(pu), o_pool[:nU], 'sharded pooled users', rtol=1e-4, atol_scale=1e-4)
            assert_close(host(pi), o_pool[nU:], 'sharded pooled items', rtol=1e-4, atol_scale=1e-4)
            assert tabs2.ws.status() == 0
            if B >= 8192 * world:
                assert getattr(tabs2, '_xchg', None) is not None and int(tabs2._inbox['idx'].abs().max()) == 0
        # ---------------- the sparse pooled-gradient exchange (marked rows pushed, masked first adjoint SpMM) ----------------
        if D == 128:
            nU2, nI2, B2, L, reg = 40000, 30000, 8192 * world, 3, 1e-5
            rng2, U2, I2, pairs2 = problem(17, nU2, nI2, D, 4 * nU2)
            lay2 = S.ShardLayout(nU2, nI2, world, rank)
            rowptr, col, val = O.build_norm_adj_csr(nU2, nI2, pairs2[:, 0], pairs2[:, 1])
            dinv = O.deg_inv_sqrt(np.diff(rowptr))
            tabs4 = S.ShardedTables(peers, lay2, D)
            tabs4.load_full(d(U2), d(I2))
            lg = S.ShardedLightGCN(tabs4, rowptr, col, dinv, L, reg, gather_first=True)
            lg.sparse_grad = True
            A = O.csr_to_torch(rowptr, col, val, nU2 + nI2)
            oU, oI = torch.from_numpy(U2.copy()), torch.from_numpy(I2.copy())
            om = [torch.zeros_like(oU), torch.zeros_like(oU), torch.zeros_like(oI), torch.zeros_like(oI)]
            for step in range(1, 3):
                sel = rng2.randint(0, len(pairs2), B2)
                user, pos = pairs2[sel, 0].astype(np.int64), pairs2[sel, 1].astype(np.int64)
                neg = rng2.randint(1, nI2 // 4, B2).astype(np.int64)          # a quarter of the items: many rows stay unmarked
                lo, hi = lay2.batch_slice(B2)
                loss = lg.step(d(user[lo:hi]), d(pos[lo:hi]), d(neg[lo:hi]), B2, 1e-3, 0.0)
                o_loss, ogU, ogI = O.lightgcn_fwd_bwd(A, oU, oI, user, pos, neg, L, reg)
                O.adam_l2_step(oU, om[0], om[1], ogU, step, 1e-3, 0.0)
                O.adam_l2_step(oI, om[2], om[3], ogI, step, 1e-3, 0.0)
                assert abs(float(loss[0]) - float(o_loss)) <= 1e-5 * abs(float(o_loss)), (float(loss[0]), float(o_loss))
                gu, gi = tabs4.gather_full()
                assert_close(host(gu), oU.numpy(), f'sparse-exchange LightGCN U step {step}', rtol=1e-4, atol_scale=1e-4)
                assert_close(host(gi), oI.numpy(), f'sparse-exchange LightGCN I step {step}', rtol=1e-4, atol_scale=1e-4)
                peers.barrier()
            assert int(lg._gm.ne(0).sum()) == 0 and tabs4.ws.status() == 0
            del lg, tabs4
        peers.host_sync()
        if rank == 0:
            print(f'dist_worker gpu ok: world {world} nU {nU} nI {nI} D {D}')
    # ---------------- the reference-facing classes on sharded tables: one ml-100k epoch against the goldens ----------------
    from tests.helpers import load, ml100k_corpus, model_args
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.BPRMF import BPRMF
    from whisprrec_b200.models.general.LightGCN import LightGCN
    from whisprrec_b200.utils import utils
    import tempfile
    corpus = ml100k_corpus()
    for cls, over, gname, tol in [(BPRMF, dict(lr=1e-3, l2=1e-6), 'ml100k_bprmf.npz', 1e-4),
                                  (LightGCN, dict(lr=2e-3, gcn_layers=2), 'ml100k_lightgcn.npz', 1e-3)]:
        g = load(gname)
        args = model_args(cls, **over)
        args.device = dev
        args.model_path = os.path.join(tempfile.gettempdir(), 'wr_dist_%s.pt' % cls.__name__)
        utils.init_seed(3407)
        model = cls(args, corpus).to(dev)
        model.fuse()
        data = {ph: cls.Dataset(model, corpus, ph) for ph in ('train', 'dev', 'test')}
        runner = BaseRunner(args)
        model.optimizer = runner._build_optimizer(model)
        model.shard(peers)
        mean_loss = runner.fit(data['train'], epoch=1)
        if 'neg_epoch1' in g.files:
            assert (data['train'].data['neg_items'] == g['neg_epoch1']).all()
        assert abs(mean_loss - float(g['epoch_mean_loss'])) <= 1e-4 * abs(float(g['epoch_mean_loss'])), mean_loss
        res = runner.evaluate(data['dev'], [10, 20], ['NDCG', 'HR'])
        for k, v in zip(g['dev_metric_keys'], g['dev_metric_vals']):
            assert abs(res[str(k)] - float(v)) <= 2e-3, (k, res[str(k)], float(v))
        model.save_model()
        ue, ie = model._embedding_pair()
        assert_close(host(ue.weight[:64]), g['after_user_rows'], 'U after a sharded epoch', rtol=tol, atol_scale=tol)
        assert_close(host(ie.weight[:64]), g['after_item_rows'], 'I after a sharded epoch', rtol=tol, atol_scale=tol)
        model.load_model()
        res2 = runner.evaluate(data['dev'], [10, 20], ['NDCG', 'HR'])
        assert res2 == res
        peers.host_sync()
        if rank == 0:
            print(f'dist_worker gpu ok: world {world} {cls.__name__} ml-100k epoch, dev', res)


if __name__ == '__main__':
    {'cpu': run_cpu, 'gpu': run_gpu}[sys.argv[1]]()
