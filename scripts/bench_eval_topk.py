#!/usr/bin/env python
"""Top-k lists at precision 2 (precision 0's lists on the tensor cores) on bench.py's configs[4]-shaped sweep point:
262,144 eval rows x 1M items, 50-item histories, D in {64, 128, 256}, k in {10, 32}.  Per (D, k) it times precision 2
with top-k, precision 2 ranks only, precision 1 with top-k (all rows) and precision 0 with top-k on a 32,768-row slice
(scaled per row), with CUDA events after a warm-up call per shape; the 0.25-1 GB item table is larger than the 126 MB L2.
It also records the list candidates per row of the last row block (mean, max), the rows rerun at precision 0 and
whether the precision-2 lists equal precision 0's on the slice.

    python scripts/bench_eval_topk.py --out-dir DIR [--reps 3]

Writes one JSON line to DIR/bench_eval_topk.json (and prints it)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from whisprrec_b200 import _lib  # noqa: E402

R, N_USERS, N_ITEMS, HIST, SLICE = 262_144, 200_000, 1_000_000, 50, 32_768
SEG_CAP = 1024                   # TC_SEG_CAP of csrc/eval_tcgen05.cu


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


def blocking():
    """exact_blocking_topk of csrc/eval_tcgen05.cu: rows per block and the rank candidate list's capacity."""
    rb = max(256, int(16e9 / N_ITEMS) // 256 * 256)
    if rb > R:
        rb = (R + 255) // 256 * 256
    cap = min(max(int(rb * N_ITEMS / 128.0), 1 << 20), 1 << 27)
    return min(rb, (1 << 30) // (SEG_CAP * 4)), cap


def segment_counts(d, scratch):
    """Candidates per row of the last row block, read back from the scratch (wr_eval_rank_tc's layout: A, B, row_ok,
    anorm, 1,024 B of counters, the rank candidate list, then the per-row segment counts)."""
    rb, cap = blocking()
    a_cols = 2 * d if d >= 256 else 3 * d
    off = align(R * a_cols * 2) + align(N_ITEMS * 3 * d * 2) + align(R) + align(R * 4) + 1024
    seg_at = align(off + cap * 8)
    last_rows = R - (R - 1) // rb * rb
    return scratch[seg_at:seg_at + 4 * last_rows].view(torch.int32)


def exact_topk_call(t, ws, scratch, k):
    U, I, user, pos, hp, hi = t
    d = U.shape[1]
    rank = torch.empty(R, dtype=torch.int32, device=U.device)
    target = torch.empty(R, dtype=torch.float32, device=U.device)
    tki = torch.empty((R, k), dtype=torch.int32, device=U.device)
    tkv = torch.empty((R, k), dtype=torch.float32, device=U.device)
    P = _lib.ptr
    _lib.check(_lib.load().wr_eval_rank_topk(P(U, _lib.F32), P(I, _lib.F32), P(user, _lib.I64), P(pos, _lib.I64), R,
                                             N_USERS, N_ITEMS, d, P(hp, _lib.I64), P(hi, _lib.I32), k, 2, P(tki, _lib.I32),
                                             P(tkv, _lib.F32), P(rank, _lib.I32), P(target, _lib.F32), None,
                                             scratch.data_ptr(), ws.ptr, _lib.stream_ptr()))
    return rank, target, tki, tkv


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out-dir', default='.')
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    ws = _lib.Workspace(dev)
    sl = slice(0, SLICE)
    out = {'what': 'full-ranking eval with top-k lists, %d rows x %d items, %d-item histories' % (R, N_ITEMS, HIST),
           'gpu': smi, 'reps': a.reps,
           'timing': 'CUDA events per call, median of reps after one warm-up call per shape; precision 0 on the first '
                     '%d rows, scaled per row' % SLICE}
    for d in (64, 128, 256):
        tabs = tables(d, dev)
        U, I, user, pos, hp, hi = tabs
        us, ps = user[sl].contiguous(), pos[sl].contiguous()
        n = _lib.load().wr_eval_scratch_bytes_topk(R, N_ITEMS, d, 2, 32)
        s = torch.empty(n + 1024, dtype=torch.uint8, device=dev)
        off = (-s.data_ptr()) % 1024
        scratch = s[off:off + n]
        for k in (10, 32):
            fns = {
                'p2_topk': lambda: exact_topk_call(tabs, ws, scratch, k),
                'p2_ranks': lambda: _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, precision=2),
                'p1_topk': lambda: _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, k=k, precision=1),
                'p0_topk_slice': lambda: _lib.eval_rank_topk(U, I, us, ps, hp, hi, ws, k=k, precision=0),
            }
            for f in fns.values():                   # warm-up: module load, tensor maps, every shape
                f()
            torch.cuda.synchronize()
            times = {name: [] for name in fns}
            for _ in range(a.reps):
                for name, f in fns.items():          # the variants alternate
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    f()
                    e1.record()
                    torch.cuda.synchronize()
                    times[name].append(e0.elapsed_time(e1))
            st = ws.status()
            med = {name: sorted(v)[len(v) // 2] for name, v in times.items()}
            r2, t2, i2, v2 = exact_topk_call(tabs, ws, scratch, k)
            cnt = segment_counts(d, scratch).to(torch.int64)
            fallback_rows = int((i2[:, 0] == -2).sum())
            st |= ws.status()
            r0, _, i0, v0, _ = _lib.eval_rank_topk(U, I, us, ps, hp, hi, ws, k=k, precision=0)
            per_row_p0 = med['p0_topk_slice'] / SLICE
            out['d%d_k%d' % (d, k)] = {
                'p2_topk_ms': med['p2_topk'], 'p2_ranks_ms': med['p2_ranks'], 'p1_topk_ms': med['p1_topk'],
                'p0_topk_slice_ms': med['p0_topk_slice'], 'p0_topk_ms_scaled_to_all_rows': per_row_p0 * R,
                'p2_topk_speedup_over_p0_topk_per_row': per_row_p0 / (med['p2_topk'] / R),
                'p2_topk_over_p2_ranks': med['p2_topk'] / med['p2_ranks'],
                'candidates_per_row_last_block_mean': float(cnt.float().mean()),
                'candidates_per_row_last_block_max': int(cnt.max()), 'segment_capacity': SEG_CAP,
                'fallback_rows': fallback_rows, 'status': st,
                'p2_lists_equal_p0_on_slice': bool(torch.equal(i2[sl], i0) and torch.equal(v2[sl], v0)),
                'p2_ranks_equal_p0_on_slice': bool(torch.equal(r2[sl], r0)),
                'all_ms': times,
            }
            print(json.dumps({'d%d_k%d' % (d, k): out['d%d_k%d' % (d, k)]}), flush=True)
        del tabs, U, I, scratch, s
        torch.cuda.empty_cache()
    line = json.dumps(out)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, 'bench_eval_topk.json'), 'w') as f:
        f.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
