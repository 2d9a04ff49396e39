#!/usr/bin/env python
"""Worker for tests/test_multi_gpu_d256.py: row-sharded tables at embedding size 256, one B200 per rank.

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29561 tests/dist_worker_d256.py

Three sharded BPRMF steps against the single-GPU step on the whole batch; item-sharded evaluation against the single-GPU
fp32 ranks at precision 0 and 2; one ml-100k epoch of BPRMF through BaseRunner on sharded tables (model.shard())
against the same epoch on one GPU, and the dev metrics of both.
"""
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.helpers import assert_close  # noqa: E402

D = 256


def main():
    from oracle import whispr_oracle as O
    from tests.helpers import ml100k_corpus, model_args
    from whisprrec_b200 import _lib
    from whisprrec_b200 import sharded as S
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.models.general.BPRMF import BPRMF
    from whisprrec_b200.utils import utils
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    assert torch.cuda.device_count() >= world, 'one GPU per rank (never share a GPU between spinning ranks)'
    peers = S.PeerGroup(dev)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    host = lambda t: t.detach().cpu().numpy()

    # ---------------- BPRMF: three sharded steps against the single-GPU step ----------------
    nU, nI, B = 1000, 3000, 4096
    rng = np.random.RandomState(5)
    U = (rng.randn(nU, D) * 0.1).astype(np.float32)
    I = (rng.randn(nI, D) * 0.1).astype(np.float32)
    pairs = np.unique(np.stack([rng.randint(0, nU, 20 * nU), rng.randint(0, nI, 20 * nU)], 1), axis=0)
    lay = S.ShardLayout(nU, nI, world, rank)
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

    # ---------------- evaluation: items sharded, ranks equal the single-GPU fp32 ranks ----------------
    half = len(pairs) // 2
    hp, hi_ = O.history_csr(nU, pairs[:half], pairs[:1])
    eu, ep = pairs[half:, 0].astype(np.int64), pairs[half:, 1].astype(np.int64)
    lh = lay.localise_history(hp, hi_)
    lh = (d(lh[0]), d(lh[1]))
    gu, gi = tabs.gather_full()
    want = _lib.eval_rank_topk(gu.contiguous(), gi.contiguous(), d(eu), d(ep), d(hp), d(hi_), ws, k=10)
    got = S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), d(eu), d(ep), lh, k=10)
    assert (host(got[0]) == host(want[0])).all(), 'sharded ranks'
    assert (host(got[1]) == host(want[1])).all(), 'sharded targets'
    assert (host(got[2]) == host(want[2])).all(), 'sharded top-k ids'
    assert (host(got[3]) == host(want[3])).all(), 'sharded top-k values'
    got2 = S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), d(eu), d(ep), lh, precision=2)
    assert (host(got2[0]) == host(want[0])).all(), 'sharded exact tensor-core ranks'
    assert tabs.ws.status() == 0 and ws.status() == 0
    peers.host_sync()
    if rank == 0:
        print(f'dist_worker_d256 ok: world {world} sharded steps and evaluation, D {D}')

    # ---------------- one ml-100k BPRMF epoch through BaseRunner: sharded against one GPU ----------------
    corpus = ml100k_corpus()
    results = []
    for sharded in (False, True):
        args = model_args(BPRMF, embedding_size=D, lr=1e-3, l2=1e-6)
        args.device = dev
        args.model_path = os.path.join(tempfile.gettempdir(), 'wr_dist_d256_%d_%d.pt' % (rank, sharded))
        utils.init_seed(3407)
        model = BPRMF(args, corpus).to(dev)
        model.fuse()
        data = {ph: BPRMF.Dataset(model, corpus, ph) for ph in ('train', 'dev')}
        runner = BaseRunner(args)
        model.optimizer = runner._build_optimizer(model)
        if sharded:
            model.shard(peers)
        mean_loss = runner.fit(data['train'], epoch=1)
        res = runner.evaluate(data['dev'], [10, 20], ['NDCG', 'HR'])
        runner.eval_precision = 0
        res0 = runner.evaluate(data['dev'], [10, 20], ['NDCG', 'HR'])
        assert res == res0, (res, res0)
        if sharded:
            model.save_model()              # gathers the shards into the reference-layout embeddings
        ue, ie = model._embedding_pair()
        results.append((mean_loss, host(ue.weight).copy(), host(ie.weight).copy(), res))
    (l1, u1, i1, r1), (l2, u2, i2, r2) = results
    assert abs(l2 - l1) <= 1e-5 * abs(l1), (l1, l2)
    assert_close(u2, u1, 'U after a sharded epoch', rtol=1e-4, atol_scale=1e-4)
    assert_close(i2, i1, 'I after a sharded epoch', rtol=1e-4, atol_scale=1e-4)
    for k in r1:
        assert abs(r1[k] - r2[k]) <= 2e-3, (k, r1[k], r2[k])
    peers.host_sync()
    if rank == 0:
        print(f'dist_worker_d256 ok: world {world} ml-100k BPRMF epoch sharded = single GPU, dev', r2)
    peers.close()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
