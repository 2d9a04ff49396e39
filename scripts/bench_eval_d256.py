#!/usr/bin/env python
"""Full-ranking evaluation at D = 256 next to D = 128, on bench.py's configs[4]-shaped sweep point (262,144 eval rows x
1M items, 50-item histories): precision 1 (ranks, and top-10), precision 2 (ranks) on all rows, precision 0 on a
32,768-row slice (a full D = 256 pass on the fp32 FMA tiles takes seconds).  The two sizes are timed alternately in one
process with CUDA events after a warm-up; the 1 GB item table alone is larger than the 126 MB L2.

    python scripts/bench_eval_d256.py --out-dir DIR [--reps 3]

Writes one JSON line to DIR/bench_eval_d256.json (and prints it)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from whisprrec_b200 import _lib  # noqa: E402

BURST_TFLOPS = 1649.7      # dense bf16 burst rate measured on one B200 (SURVEY.md, section on measured peaks)
R, N_USERS, N_ITEMS, HIST, SLICE = 262_144, 200_000, 1_000_000, 50, 32_768


def align(x, a=1024):
    return (x + a - 1) // a * a


def tables(d, dev):
    g = torch.Generator(device=dev)
    g.manual_seed(3407)
    U = torch.randn((N_USERS, d), device=dev, generator=g) / d ** 0.5
    I = torch.randn((N_ITEMS, d), device=dev, generator=g)
    user = torch.randint(0, N_USERS, (R,), device=dev, generator=g)
    pos = torch.randint(0, N_ITEMS, (R,), device=dev, generator=g)
    hp = torch.arange(0, (N_USERS + 1) * HIST, HIST, device=dev, dtype=torch.int64)
    hi = torch.sort(torch.randint(0, N_ITEMS, (N_USERS, HIST), device=dev, generator=g), dim=1).values
    return U, I, user, pos, hp, hi.to(torch.int32).reshape(-1).contiguous()


def exact_call(t, ws, scratch):
    """precision 2 through the C entry point with our own scratch, so the candidate count of the last row block can be
    read back (wr_eval_rank_tc's layout: A, B, row_ok, anorm, then bmax at +0 and the count at +16)."""
    U, I, user, pos, hp, hi = t
    d = U.shape[1]
    rank = torch.empty(R, dtype=torch.int32, device=U.device)
    target = torch.empty(R, dtype=torch.float32, device=U.device)
    P = _lib.ptr
    _lib.check(_lib.load().wr_eval_rank_topk(P(U, _lib.F32), P(I, _lib.F32), P(user, _lib.I64), P(pos, _lib.I64), R,
                                             N_USERS, N_ITEMS, d, P(hp, _lib.I64), P(hi, _lib.I32), 0, 2, None, None,
                                             P(rank, _lib.I32), P(target, _lib.F32), None, scratch.data_ptr(), ws.ptr,
                                             _lib.stream_ptr()))
    return rank


def candidate_fraction(d, scratch):
    a_cols = 2 * d if d >= 256 else 3 * d
    off = align(R * a_cols * 2) + align(N_ITEMS * 3 * d * 2) + align(R) + align(R * 4) + 16
    cnt = int(scratch[off:off + 8].view(torch.int64).item())
    rb = max(256, int(16e9 / N_ITEMS) // 256 * 256)
    if rb > R:
        rb = (R + 255) // 256 * 256
    last_rows = R - (R - 1) // rb * rb
    return cnt / (last_rows * N_ITEMS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out-dir', default='.')
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dims = (128, 256)
    tabs = {d: tables(d, dev) for d in dims}
    ws = _lib.Workspace(dev)
    scratch = {}
    for d in dims:
        n = _lib.load().wr_eval_scratch_bytes(R, N_ITEMS, d, 2)
        s = torch.empty(n + 1024, dtype=torch.uint8, device=dev)
        off = (-s.data_ptr()) % 1024
        scratch[d] = s[off:off + n]
    sl = slice(0, SLICE)

    def runs(d):
        U, I, user, pos, hp, hi = tabs[d]
        us, ps = user[sl].contiguous(), pos[sl].contiguous()
        return {
            'p1': lambda: _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, precision=1),
            'p1_top10': lambda: _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, precision=1, k=10),
            'p2': lambda: exact_call(tabs[d], ws, scratch[d]),
            'p0_slice': lambda: _lib.eval_rank_topk(U, I, us, ps, hp, hi, ws, precision=0),
        }
    fns = {d: runs(d) for d in dims}
    for d in dims:                                   # warm-up: module load, tensor maps, every shape
        for f in fns[d].values():
            f()
    torch.cuda.synchronize()
    times = {d: {k: [] for k in fns[d]} for d in dims}
    for _ in range(a.reps):
        for d in dims:                               # the two sizes alternate
            for k, f in fns[d].items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                torch.cuda.synchronize()
                times[d][k].append(e0.elapsed_time(e1))
    assert ws.status() == 0, ws.status()
    out = {'what': 'full-ranking eval, %d rows x %d items, %d-item histories, k = 0 unless noted' % (R, N_ITEMS, HIST),
           'gpu': smi, 'reps': a.reps, 'timing': 'CUDA events per call, median of reps after one warm-up call per shape',
           'burst_tflops': BURST_TFLOPS, 'burst_note': 'fraction of the measured 1,649.7 TFLOP/s dense bf16 burst'}
    for d in dims:
        med = {k: sorted(v)[len(v) // 2] for k, v in times[d].items()}
        useful = 2.0 * R * N_ITEMS * d
        useful_slice = 2.0 * SLICE * N_ITEMS * d
        U, I, user, pos, hp, hi = tabs[d]
        r2 = exact_call(tabs[d], ws, scratch[d])
        frac = candidate_fraction(d, scratch[d])
        r0 = _lib.eval_rank_topk(U, I, user[sl].contiguous(), pos[sl].contiguous(), hp, hi, ws, precision=0)[0]
        p1_tf = useful / (med['p1'] * 1e-3) / 1e12
        p2_tf = useful / (med['p2'] * 1e-3) / 1e12
        p0_tf = useful_slice / (med['p0_slice'] * 1e-3) / 1e12
        out['d%d' % d] = {
            'p1_ms': med['p1'], 'p1_tflops': p1_tf, 'p1_frac_of_burst': p1_tf / BURST_TFLOPS,
            'p1_top10_ms': med['p1_top10'], 'p1_top10_tflops': useful / (med['p1_top10'] * 1e-3) / 1e12,
            'p2_ms': med['p2'], 'p2_useful_tflops': p2_tf, 'p2_tensor_tflops': 3 * p2_tf,
            'p2_tensor_frac_of_burst': 3 * p2_tf / BURST_TFLOPS,
            'p2_recheck_candidate_fraction_last_row_block': frac,
            'p0_slice_rows': SLICE, 'p0_slice_ms': med['p0_slice'], 'p0_tflops': p0_tf,
            'p2_speedup_over_p0_per_row': (med['p0_slice'] / SLICE) / (med['p2'] / R),
            'p2_ranks_equal_p0_on_slice': bool(torch.equal(r0, r2[sl])),
            'all_ms': times[d],
        }
        assert ws.status() == 0, ws.status()
    line = json.dumps(out)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, 'bench_eval_d256.json'), 'w') as f:
        f.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
