#!/usr/bin/env python
"""Where the time of one single-launch BPRMF step (bprmf_step_kernel, wr_bprmf_step) goes with a cold L2.

    python scripts/prof_step_phases.py [--lib PATH.so ...] [--reps N] [--out out.json]

Bench shape: 6,040 x 3,706 rows, D = 64, B = 2048, a 512 MB buffer written between steps (outside the events).  For each
library (default: the in-tree build) it reports
  * the event-timed step beside the event floor (a 4-element Adam sweep timed the same way, after the same flush);
  * from the traced instantiation (wr_debug_step_trace: %globaltimer stamps of thread 0 of every CTA), per phase, the
    median over steps of the median over CTAs (`median_cta`) and the critical path (`critical`: the latest CTA at each
    stamp, measured from the earliest entry).  Stamp 1 (`ids_mv_prefetch`) is thread 0's first ids landed, with the
    G / M / V prefetch that waits for them issued.
Several --lib arguments compare builds in one process (each is loaded in a child process of its own).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
STAMPS = ['entry', 'ids_mv_prefetch', 'rows', 'reds_issued', 'arrived', 'passed', 'adam_operands', 'exit']
PHASES = [('launch_to_ids', 0, 1), ('ids_to_rows', 1, 2), ('rows_to_reds', 2, 3), ('fence_and_arrive', 3, 4),
          ('barrier_wait', 4, 5), ('adam_operands', 5, 6), ('adam_to_exit', 6, 7)]


def measure(reps):
    import torch
    from whisprrec_b200 import _lib
    nU, nI, D, B = 6040, 3706, 64, 2048
    dev = torch.device('cuda')
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    P = torch.randn((nU + nI, D), device=dev, generator=g) * 0.1
    M, V, G = torch.zeros_like(P), torch.zeros_like(P), torch.zeros_like(P)
    ws, loss = _lib.Workspace(dev), torch.zeros(1, device=dev)
    u = torch.randint(0, nU, (B,), device=dev, generator=g)
    p = torch.randint(0, nI, (B,), device=dev, generator=g)
    n = torch.randint(1, nI, (B,), device=dev, generator=g)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    tiny = [torch.zeros(4, device=dev) for _ in range(4)]
    lib = _lib.load()
    k = [0]

    def step():
        k[0] += 1
        _lib.bprmf_step(P, M, V, G, u, p, n, nU, k[0], 1e-3, 1e-6, loss, ws)

    def ev_time(fn):
        ms = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1) * 1e3)
        return {'median': float(np.median(ms)), 'mean': float(np.mean(ms)), 'min': float(np.min(ms))}

    out = {'lib': _lib.LIB_PATH, 'gpu': torch.cuda.get_device_name(0)}
    floor = lambda: _lib.adam_l2_sweep(*tiny, 1, 1e-3, 0.0)
    for name, fn in (('floor_tiny_kernel_us', floor), ('step_us', step)):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        out[name] = ev_time(fn)
    trace = torch.zeros((2048, 8), dtype=torch.int64, device=dev)
    _lib.check(lib.wr_debug_step_trace(trace.data_ptr()))
    step(); torch.cuda.synchronize()
    out['traced_step_us'] = ev_time(step)
    per_cta, crit = [], []
    for _ in range(reps):
        trace.zero_()
        flush.zero_()
        step()
        torch.cuda.synchronize()
        t = trace.cpu().numpy()
        t = t[t[:, 0] != 0].astype(np.int64)            # [grid, 8]
        assert (np.diff(t, axis=1) >= 0).all(), 'stamps decrease within a CTA'
        per_cta.append([np.median(t[:, b] - t[:, a]) for _, a, b in PHASES])
        crit.append(t.max(0) - t[:, 0].min())
    _lib.check(lib.wr_debug_step_trace(None))
    out['grid'] = int(t.shape[0])
    out['single_step_flushed_phases_ns'] = {
        'median_cta': {name: float(np.median([r[q] for r in per_cta])) for q, (name, _, _) in enumerate(PHASES)},
        'critical': {s: float(np.median([c[q] for c in crit])) for q, s in enumerate(STAMPS)},
        'note': 'median_cta: median over steps of the median over CTAs of each phase; critical: latest CTA at each stamp, '
                'from the earliest entry'}
    assert ws.status() == 0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--lib', action='append', default=[])
    ap.add_argument('--reps', type=int, default=100)
    ap.add_argument('--out', default=None)
    ap.add_argument('--child', action='store_true', help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        if a.lib:
            from whisprrec_b200 import _lib
            _lib.LIB_PATH = os.path.abspath(a.lib[0])
        print(json.dumps(measure(a.reps)))
        return
    res = {}
    for lib in a.lib or [None]:
        cmd = [sys.executable, os.path.abspath(__file__), '--child', '--reps', str(a.reps)] + (['--lib', lib] if lib else [])
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
        if r.returncode != 0:
            sys.stderr.write(r.stderr[-3000:])
            raise SystemExit('measuring %s failed' % (lib or 'the in-tree build'))
        res[lib or 'in-tree'] = json.loads(r.stdout.strip().splitlines()[-1])
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True).stdout.strip()
    except OSError:
        q = None
    res['card'] = q
    print(json.dumps(res, indent=1))
    if a.out:
        json.dump(res, open(a.out, 'w'), indent=1)


if __name__ == '__main__':
    main()
