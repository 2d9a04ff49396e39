#!/usr/bin/env python
"""Worker for tests/test_multi_gpu_topk_long.py: item-sharded top-k lists of 100 items, one B200 per rank.

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29564 tests/dist_worker_topk_long.py

sharded_eval(..., k=100) at precisions 2 and 0 (local long lists, all-gather, wr_topk_merge_long) against single-GPU
precision 0 at D = 64 and 256: ranks, targets and the lists (ids and values) equal on every rank.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from oracle import whispr_oracle as O
    from whisprrec_b200 import _lib
    from whisprrec_b200 import sharded as S
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    assert torch.cuda.device_count() >= world, 'one GPU per rank (never share a GPU between spinning ranks)'
    peers = S.PeerGroup(dev)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    host = lambda t: t.detach().cpu().numpy()
    ws = _lib.Workspace(dev)
    for D in (64, 256):
        nU, nI = 2000, 30_000
        rng = np.random.RandomState(D)
        U = (rng.randn(nU, D) / np.sqrt(D)).astype(np.float32)
        I = (rng.randn(nI, D) * rng.uniform(0.5, 1.5, (nI, 1))).astype(np.float32)
        I[7] = I[3]
        U[11] = 0.0
        pairs = np.unique(np.stack([rng.randint(0, nU, 30 * nU), rng.randint(0, nI, 30 * nU)], 1), axis=0)
        half = len(pairs) // 2
        hp, hi_ = O.history_csr(nU, pairs[:half], pairs[:1])
        eu, ep = pairs[half:, 0].astype(np.int64), pairs[half:, 1].astype(np.int64)
        lay = S.ShardLayout(nU, nI, world, rank)
        tabs = S.ShardedTables(peers, lay, D)
        tabs.load_full(d(U), d(I))
        lh = lay.localise_history(hp, hi_)
        lh = (d(lh[0]), d(lh[1]))
        gu, gi = tabs.gather_full()
        want = _lib.eval_rank_topk(gu.contiguous(), gi.contiguous(), d(eu), d(ep), d(hp), d(hi_), ws, k=100, precision=0)
        for precision in (2, 0):
            got = S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), d(eu), d(ep), lh, k=100, precision=precision)
            for g, w, what in zip(got, want, ('ranks', 'targets', 'top-k ids', 'top-k values')):
                assert (host(g) == host(w)).all(), (D, precision, what)
            assert tabs.ws.status() == 0 and ws.status() == 0
            assert tabs.ws.last_topk_fallback_rows == 0
        peers.host_sync()
        if rank == 0:
            print(f'dist_worker_topk_long ok: world {world} D {D} sharded top-100 = precision 0')
    peers.close()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
