#!/usr/bin/env python
"""Row-sharded SGL training step on the shapes of scripts/bench_sgl_scale.py, one process per GPU.

    python -m torch.distributed.run --nproc-per-node 8 scripts/bench_sgl_sharded.py --out profiles/r08_bench_sgl_sharded.json

World 1 runs the same sharded code on one GPU (torchrun --nproc-per-node 1).  For each shape, on every rank:
  * parity: the first step on the first batch against the single-GPU SGL.predict + FusedAdam step on the same tables,
    views and batch (rank 0 builds that model too): the batch loss and the ego gradient before Adam;
  * the step time over whole steps (CUDA events, no events inside; at least --steps steps and --min-window-ms of work,
    the batches reused in turn), then the same steps with an event at each phase boundary -- ShardedSGL.step's own
    `mark` hook: the three propagations, BPR + EmbLoss norms, InfoNCE users, InfoNCE items, the three adjoints, EmbLoss
    scatter, Adam -- and the time spent in the cross-GPU barriers (an event pair around each), medians over the steps.
Rank 0 writes the JSON (one entry per shape, with the GPU name, power limit and max SM clock read in the same run);
when --out names an existing file from other world sizes, the entries are merged by (world, shape).
"""
import argparse
import json
import os
import random
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

from bench_sgl_scale import SHAPES, _Corpus, gpu_info  # noqa: E402
from whisprrec_b200 import _lib  # noqa: E402
from whisprrec_b200 import sharded as S  # noqa: E402
from whisprrec_b200.main import default_args  # noqa: E402
from whisprrec_b200.models.BaseModel import FusedAdam  # noqa: E402
from whisprrec_b200.models.general.SGL import SGL  # noqa: E402
from whisprrec_b200.utils import synthetic  # noqa: E402

PHASES = ('propagate_x3', 'bpr_embloss_norms', 'infonce_users', 'infonce_items', 'adjoint_x3', 'embloss_scatter', 'adam')


def bench_shape(name, n_users, n_items, n_inter, a, peers):
    dev, world, rank = peers.device, peers.world, peers.rank
    t0 = time.time()
    u, i = synthetic.power_law_pairs(n_users, n_items, n_inter, seed=3407, device=dev)
    corpus = _Corpus(n_users, n_items, u.cpu().numpy(), i.cpu().numpy())
    del u, i
    args = default_args(SGL, embedding_size=a.dim, batch_size=a.batch, lr=1e-3, l2=0.0)

    def make_model():
        torch.manual_seed(3407)
        m = SGL(args, corpus).to(dev)
        m.fuse()
        m.optimizer = FusedAdam(m, args.lr, args.l2)
        return m
    rng = np.random.RandomState(0)
    E = len(corpus.users)
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.int64)).to(dev)
    steps = a.steps if n_users + n_items < 500_000 else max(3, a.steps // 4)
    batches = []
    for _ in range(1 + a.warmup + steps):
        sel = rng.randint(0, E, a.batch)
        batches.append(torch.stack([d(corpus.users[sel]), d(corpus.items[sel]), d(rng.randint(0, n_items, a.batch))]))
    B = a.batch
    parity = None
    if rank == 0:                       # the single-GPU step on the first batch
        ref = make_model()
        random.seed(11)
        ref.graph_construction()
        b = batches[0]
        ref.predict({'user_id': b[0], 'pos_item': b[1], 'neg_items': b[2]})
        ref_loss, ref_G = float(ref.tables.loss.item()), ref.tables.G.clone()
        ref.optimizer.step()
        del ref
        torch.cuda.empty_cache()
    model = make_model()
    st = model.shard(peers)
    g = model.sharded_sgl
    lay = st.layout
    random.seed(11)
    model.graph_construction()
    grad, grad_s = st.symmetric()
    adam = st.adam
    st.adam = lambda *x, **k: (grad.copy_(st.G), adam(*x, **k))
    lo, hi = lay.batch_slice(B)
    b = batches[0]
    loss = float(model.sharded_train_step(b[0, lo:hi], b[1, lo:hi], b[2, lo:hi], B, args.lr, 0.0, batch=b)[0])
    st.adam = adam
    gu, gi = st.gather_full(grad_s)
    if rank == 0:
        G = torch.cat([gu, gi])
        parity = {'loss': loss, 'loss_single_gpu': ref_loss, 'loss_rel_diff': abs(loss - ref_loss) / abs(ref_loss),
                  'grad_maxdiff_over_max': float((G - ref_G).abs().max() / ref_G.abs().max())}
        parity['ok'] = parity['loss_rel_diff'] <= 1e-5 and parity['grad_maxdiff_over_max'] <= 1e-4
        del ref_G, G
    del gu, gi
    setup_s = time.time() - t0

    def step(b, mark=None):
        return g.step(b[0, lo:hi], b[1, lo:hi], b[2, lo:hi], B, args.lr, 0.0, b[0], b[1], mark=mark)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for b in batches[1:1 + a.warmup]:
        step(b)
    e1.record()
    torch.cuda.synchronize()
    # enough steps for a window of at least min_window_ms (the same count on every rank: the largest estimate wins)
    est = torch.tensor([e0.elapsed_time(e1) / a.warmup])
    dist.all_reduce(est, op=dist.ReduceOp.MAX)
    steps = max(steps, int(np.ceil(a.min_window_ms / float(est[0]))))
    timed = [batches[1 + a.warmup + k % (len(batches) - 1 - a.warmup)] for k in range(steps)]
    peers.host_sync()
    e0.record()
    for b in timed:
        step(b)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    # the same steps with an event after each phase and an event pair around each barrier
    barrier = st.peers.barrier
    pairs = []

    def timed_barrier(*x, **k):
        be = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        be[0].record()
        out = barrier(*x, **k)
        be[1].record()
        pairs.append(be)
        return out
    st.peers.barrier = timed_barrier
    split = {k: [] for k in PHASES}
    barrier_ms, n_barriers = [], 0
    peers.host_sync()
    for b in timed:
        ev = {'start': torch.cuda.Event(enable_timing=True)}
        ev['start'].record()

        def mark(name):
            ev[name] = torch.cuda.Event(enable_timing=True)
            ev[name].record()
        pairs.clear()
        step(b, mark)
        torch.cuda.synchronize()
        names = ['start'] + list(PHASES)
        assert list(ev) == names, list(ev)          # the phases ShardedSGL.step marks, in this order
        for k, ph in enumerate(PHASES):
            split[ph].append(ev[names[k]].elapsed_time(ev[ph]))
        barrier_ms.append(sum(x.elapsed_time(y) for x, y in pairs))
        n_barriers = len(pairs)
    st.peers.barrier = barrier
    split = {k: float(np.median(v)) for k, v in split.items()}
    st.ws.raise_on_status()
    D = a.dim
    n_local = {'users': len(lay.local_users()), 'items': len(lay.local_items())}
    out = {
        'shape': name, 'world': world, 'users': n_users, 'items': n_items, 'interactions': E, 'dim': D, 'batch': B,
        'gcn_layers': g.L, 'steps': steps, 'ms_per_step': step_ms, 'phase_ms_median': split,
        'phase_sum_ms': float(sum(split.values())), 'barrier_ms_median': float(np.median(barrier_ms)),
        'barriers_per_step': n_barriers,
        'infonce_share_of_phases': (split['infonce_users'] + split['infonce_items']) / sum(split.values()),
        'infonce_tflops_per_gpu_8BND_local': {
            'infonce_users': 8.0 * B * n_local['users'] * D / (split['infonce_users'] * 1e-3) / 1e12,
            'infonce_items': 8.0 * B * n_local['items'] * D / (split['infonce_items'] * 1e-3) / 1e12},
        # z partials to the world - 1 peers; the batch's T1 / T2 rows gathered and its Ga partials stored, (world - 1) / world
        # of them remote
        'infonce_nvlink_bytes_per_rank_per_block': 4 * B * (world - 1) + 3 * 4 * B * D * (world - 1) // world,
        'gather_first': g.gather_first, 'setup_s': setup_s, 'mem_gb': torch.cuda.max_memory_allocated(dev) / 1e9,
        'parity_first_step': parity,
    }
    del model, g, st
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--dim', type=int, default=64)
    ap.add_argument('--batch', type=int, default=2048)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--min-window-ms', type=float, default=2000.0, help='time at least this much work per shape')
    ap.add_argument('--shapes', default=','.join(k for k in SHAPES if not k.startswith('ml-1m')))
    ap.add_argument('--out', default=None, help='write / merge the JSON here (rank 0)')
    a = ap.parse_args()
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dist.init_process_group('gloo')
    peers = S.PeerGroup(torch.device('cuda', local))
    info = gpu_info() if peers.rank == 0 else {}
    lines = []
    for name in a.shapes.split(','):
        line = bench_shape(name, *SHAPES[name], a, peers)
        if peers.rank == 0:
            print(json.dumps(line), flush=True)
            lines.append(line)
    peers.close()
    if peers.rank == 0 and a.out:
        result = {'bench': 'row-sharded SGL step (scripts/bench_sgl_sharded.py)', **info, 'runs': []}
        if os.path.exists(a.out):
            with open(a.out) as f:
                result['runs'] = json.load(f).get('runs', [])
        keep = {(l['world'], l['shape']) for l in lines}
        result['runs'] = [r for r in result['runs'] if (r['world'], r['shape']) not in keep] + lines
        result['runs'].sort(key=lambda r: (r['shape'], r['world']))
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(result, f, indent=1)
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
