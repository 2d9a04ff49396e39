#!/usr/bin/env python
"""SGL training step on synthetic corpora shaped like the public SGL / LightGCN datasets, one GPU.

    python scripts/bench_sgl_scale.py --out profiles/r07_bench_sgl_scale.json
    python scripts/bench_sgl_scale.py --baseline-lib /path/to/other/libwhisprrec_b200.so ...

For each shape: the step time of SGL.predict + FusedAdam (CUDA events) and its split into the three propagations, the
BPR term, the two InfoNCE calls, the three adjoint propagations, EmbLoss and Adam (events between the phases of one
step, on the same stream); the InfoNCE rate counted as 8 B N D flop (pass 1 computes the scores once, pass 2 again for
the two gradient products).  With --baseline-lib (a libwhisprrec_b200.so built from another commit, e.g. the parent's
`make -C whisprrec_b200/csrc` in a `git worktree`), the two libraries' InfoNCE calls are alternated in the same process on
the ml-1m-shaped tables, and their outputs compared.

The corpora are utils/synthetic.power_law_pairs with the user / item / interaction counts of the named dataset; results
are labelled "<name>-shaped synthetic", never by the dataset's name.  The GPU's name, power limit and max SM clock are
read with nvidia-smi in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from whisprrec_b200 import _lib  # noqa: E402
from whisprrec_b200.main import default_args  # noqa: E402
from whisprrec_b200.models.general.SGL import SGL  # noqa: E402
from whisprrec_b200.utils import synthetic  # noqa: E402

SHAPES = {
    'ml-1m-shaped synthetic': (6040, 3706, 1_000_209),
    'Amazon-Book-shaped synthetic': (52_643, 91_599, 2_984_108),
    'Alibaba-iFashion-shaped synthetic': (300_000, 81_614, 1_607_813),
    '1M x 200k power-law synthetic': (1_000_000, 200_000, 5_000_000),
}
PHASES = ('propagate_x3', 'bpr', 'infonce_users', 'infonce_items', 'adjoint_x3', 'embloss', 'adam')


class _Corpus(object):
    """What SGL needs from a reader: the counts and the training CSR."""

    def __init__(self, n_users, n_items, users, items):
        self.n_users, self.n_items = n_users, n_items
        code = np.unique(users.astype(np.int64) * n_items + items)
        uu, ii = code // n_items, code % n_items
        ptr = np.zeros(n_users + 1, dtype=np.int64)
        np.cumsum(np.bincount(uu, minlength=n_users), out=ptr[1:])
        self._csr = (ptr, ii.astype(np.int32))
        self.users, self.items = uu, ii

    def train_csr(self):
        return self._csr


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.splitlines()[0].split(','))
    return {'gpu': name, 'power_limit': power, 'max_sm_clock': clock}


def phased_step(model, user, pos, neg, ev):
    """SGL.predict + FusedAdam.step with an event after each phase (the same kernels in the same order)."""
    t = model.tables
    model._prepare_grads()
    out = t.loss
    L = model.gcn_layers
    graphs = [model.train_graph] + model.sub_graphs
    ev[0].record()
    for g, pool in zip(graphs, model.pool):
        model._propagate(g, pool)
    ev[1].record()
    scale = 1.0 / (L + 1)
    pm, gm = model.pool[0], model.pool_grad[0]
    _lib.bpr_logsig_sum_fwd_bwd(t.users(pm), t.items(pm), user, pos, neg, t.users(gm), t.items(gm), out, t.ws,
                                grad_scale=scale)
    ev[2].record()
    p1, p2, g1, g2 = model.pool[1], model.pool[2], model.pool_grad[1], model.pool_grad[2]
    model._scratch = _lib.infonce_fwd_bwd(t.users(p1), t.users(p2), user, model.ssl_tau, model.ssl_weight, scale,
                                          t.users(g1), t.users(g2), out, t.ws, model._scratch)
    ev[3].record()
    model._scratch = _lib.infonce_fwd_bwd(t.items(p1), t.items(p2), pos, model.ssl_tau, model.ssl_weight, scale,
                                          t.items(g1), t.items(g2), out, t.ws, model._scratch)
    ev[4].record()
    for n, (g, grad) in enumerate(zip(graphs, model.pool_grad)):
        model._adjoint(g, grad, first=n == 0)
    ev[5].record()
    _lib.embloss_fwd_bwd(t.users(t.P), t.items(t.P), user, pos, neg, t.users(t.G), t.items(t.G), out, t.ws,
                         model.reg_weight)
    ev[6].record()
    model.optimizer.step()
    ev[7].record()


def bench_shape(name, n_users, n_items, n_inter, a, dev):
    t0 = time.time()
    u, i = synthetic.power_law_pairs(n_users, n_items, n_inter, seed=3407, device=dev)
    corpus = _Corpus(n_users, n_items, u.cpu().numpy(), i.cpu().numpy())
    args = default_args(SGL, embedding_size=a.dim, batch_size=a.batch, lr=1e-3, l2=0.0)
    torch.manual_seed(3407)
    model = SGL(args, corpus).to(dev)
    model.fuse()
    from whisprrec_b200.models.BaseModel import FusedAdam
    model.optimizer = FusedAdam(model, args.lr, args.l2)
    model.graph_construction()
    torch.cuda.synchronize()
    setup_s = time.time() - t0
    rng = np.random.RandomState(0)
    E = len(corpus.users)

    def batch():
        sel = rng.randint(0, E, a.batch)
        d = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.int64)).to(dev)
        return d(corpus.users[sel]), d(corpus.items[sel]), d(rng.randint(0, n_items, a.batch))

    steps = a.steps if n_users + n_items < 500_000 else max(3, a.steps // 4)
    batches = [batch() for _ in range(a.warmup + steps)]
    for b in batches[:a.warmup]:
        model.predict({'user_id': b[0], 'pos_item': b[1], 'neg_items': b[2]})
        model.optimizer.step()
    torch.cuda.synchronize()
    # whole steps, no events inside
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for b in batches[a.warmup:]:
        model.predict({'user_id': b[0], 'pos_item': b[1], 'neg_items': b[2]})
        model.optimizer.step()
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    # the same steps with an event after each phase
    split = {k: [] for k in PHASES}
    for b in batches[a.warmup:]:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
        phased_step(model, b[0], b[1], b[2], ev)
        torch.cuda.synchronize()
        for k, name_ in enumerate(PHASES):
            split[name_].append(ev[k].elapsed_time(ev[k + 1]))
    split = {k: float(np.median(v)) for k, v in split.items()}
    loss = float(model.tables.loss.item())
    st = model.tables.ws.status()
    D, B = a.dim, a.batch
    fl = {'infonce_users': 8.0 * B * n_users * D, 'infonce_items': 8.0 * B * n_items * D}
    out = {
        'shape': name, 'users': n_users, 'items': n_items, 'interactions': E, 'dim': D, 'batch': B,
        'gcn_layers': model.gcn_layers, 'steps': steps, 'ms_per_step': step_ms,
        'phase_ms_median': split, 'phase_sum_ms': float(sum(split.values())),
        'infonce_share_of_phases': (split['infonce_users'] + split['infonce_items']) / sum(split.values()),
        'infonce_flop_counted': '8 B N D per call',
        'infonce_tflops': {k: fl[k] / (split[k] * 1e-3) / 1e12 for k in fl},
        'infonce_scratch_mb': _lib.load().wr_infonce_scratch_bytes(B, max(n_users, n_items), D) / 2 ** 20,
        'last_loss': loss, 'finite_loss': bool(np.isfinite(loss)), 'status': st, 'setup_s': setup_s,
        'mem_gb': torch.cuda.max_memory_allocated() / 1e9,
    }
    return out, model


def _attach(path):
    """The InfoNCE entry points of another build of the library."""
    lib = ctypes.CDLL(path)
    for name in ('wr_workspace_bytes', 'wr_workspace_init', 'wr_infonce_scratch_bytes', 'wr_infonce_fwd_bwd'):
        res, args = _lib.SIGNATURES[name]
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def compare_with_baseline(model, a, dev):
    """The parent-or-other library's InfoNCE against this one on the ml-1m-shaped pooled views, alternated."""
    t = model.tables
    stream = _lib.stream_ptr()
    libs = {'new': _lib.load(), 'baseline': _attach(a.baseline_lib)}
    rng = np.random.RandomState(7)
    res = {}
    for term, (T1, T2, nrows) in {'users': (t.users(model.pool[1]), t.users(model.pool[2]), t.n_users),
                                  'items': (t.items(model.pool[1]), t.items(model.pool[2]), t.n_items)}.items():
        N, D = T1.shape
        idx = torch.from_numpy(rng.randint(0, nrows, a.batch).astype(np.int64)).to(dev)
        state = {}
        for k, lib in libs.items():
            wsb = torch.empty(lib.wr_workspace_bytes(), dtype=torch.uint8, device=dev)
            _lib.check(lib.wr_workspace_init(wsb.data_ptr(), stream))
            nb = lib.wr_infonce_scratch_bytes(a.batch, N, D)
            state[k] = dict(ws=wsb, scratch=torch.empty(nb, dtype=torch.uint8, device=dev), scratch_mb=nb / 2 ** 20,
                            g1=torch.zeros_like(T1), g2=torch.zeros_like(T2), loss=torch.zeros(1, device=dev))

        def call(k):
            s, lib = state[k], libs[k]
            _lib.check(lib.wr_infonce_fwd_bwd(T1.data_ptr(), T2.data_ptr(), idx.data_ptr(), a.batch, N, D, model.ssl_tau,
                                              model.ssl_weight, 1.0 / 3, s['g1'].data_ptr(), s['g2'].data_ptr(),
                                              s['loss'].data_ptr(), s['scratch'].data_ptr(), s['scratch'].numel(),
                                              s['ws'].data_ptr(), stream))
        for k in libs:                                   # one call each on zeroed outputs for the comparison
            call(k)
        torch.cuda.synchronize()
        g = {k: (float(state[k]['loss'].item()), state[k]['g1'].clone(), state[k]['g2'].clone()) for k in libs}
        for k in libs:
            for _ in range(3):
                call(k)
        times = {k: [] for k in libs}
        for _ in range(a.rounds):
            for k in libs:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.reps):
                    call(k)
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.reps)
        rel = lambda x, y: float((x - y).abs().max() / y.abs().max())
        med = {k: float(np.median(v)) for k, v in times.items()}
        res[term] = {
            'B': a.batch, 'N': N, 'D': D, 'ms_median': med, 'ms_all': times,
            'speedup_new_over_baseline': med['baseline'] / med['new'],
            'new_tflops_8BND': 8.0 * a.batch * N * D / (med['new'] * 1e-3) / 1e12,
            'baseline_tflops_6BND': 6.0 * a.batch * N * D / (med['baseline'] * 1e-3) / 1e12,
            'scratch_mb': {k: state[k]['scratch_mb'] for k in libs},
            'loss': {k: g[k][0] for k in libs}, 'loss_rel_diff': abs(g['new'][0] - g['baseline'][0]) / abs(g['baseline'][0]),
            'dT1_maxdiff_over_max': rel(g['new'][1], g['baseline'][1]),
            'dT2_maxdiff_over_max': rel(g['new'][2], g['baseline'][2]),
            'status': {k: int(state[k]['ws'][:4].view(torch.int32).item()) for k in libs},
        }
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--dim', type=int, default=64)
    ap.add_argument('--batch', type=int, default=2048)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--shapes', default=','.join(SHAPES), help='comma-separated names from SHAPES')
    ap.add_argument('--baseline-lib', default=None, help='another build of libwhisprrec_b200.so to alternate with')
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None, help='write the JSON here as well as to stdout')
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    result = {'bench': 'SGL step on synthetic corpora (scripts/bench_sgl_scale.py)', **gpu_info(), 'shapes': []}
    for name in a.shapes.split(','):
        line, model = bench_shape(name, *SHAPES[name], a, dev)
        if a.baseline_lib and name.startswith('ml-1m'):
            line['infonce_vs_baseline'] = compare_with_baseline(model, a, dev)
        result['shapes'].append(line)
        print(json.dumps(line), flush=True)
        del model
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
