#!/usr/bin/env python
"""Top-k lists of up to 256 items (wr_eval_rank_topk_long) on bench.py's configs[4]-shaped sweep point: 262,144 eval
rows x 1M items, 50-item histories, D in {64, 128, 256}, k in {32, 64, 100, 256}.  k = 32 is the existing
wr_eval_rank_topk path, timed as the reference.  Per (D, k) it times precision-2 lists, precision-2 ranks only and
precision-0 lists on a 32,768-row slice (scaled per row), with CUDA events after a warm-up call per shape; the
0.25-1 GB item table is larger than the 126 MB L2.  It also records the candidates per row of the last row block
(mean, max), the rows the sweep finished and whether the precision-2 lists equal precision 0's on the slice.

    python scripts/bench_eval_topk_long.py --out-dir DIR [--reps 3]

Writes one JSON line to DIR/bench_eval_topk_long.json (and prints it)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from whisprrec_b200 import _lib  # noqa: E402
from scripts.bench_eval_topk import R, N_USERS, N_ITEMS, HIST, SLICE, align, exact_topk_call, tables  # noqa: E402

RANGES, LONG_ROWS = 16, 65_536       # WR_LONG_RANGES, WR_LONG_BLOCK_ROWS of csrc/common.cuh


def long_call(t, ws, scratch, k, precision):
    U, I, user, pos, hp, hi = t
    n, d = user.numel(), U.shape[1]
    rank = torch.empty(n, dtype=torch.int32, device=U.device)
    target = torch.empty(n, dtype=torch.float32, device=U.device)
    tki = torch.empty((n, k), dtype=torch.int32, device=U.device)
    tkv = torch.empty((n, k), dtype=torch.float32, device=U.device)
    P = _lib.ptr
    _lib.check(_lib.load().wr_eval_rank_topk_long(P(U, _lib.F32), P(I, _lib.F32), P(user, _lib.I64), P(pos, _lib.I64),
                                                  n, N_USERS, N_ITEMS, d, P(hp, _lib.I64), P(hi, _lib.I32), k, precision,
                                                  P(tki, _lib.I32), P(tkv, _lib.F32), P(rank, _lib.I32),
                                                  P(target, _lib.F32), scratch.data_ptr(), ws.ptr, _lib.stream_ptr()))
    return rank, target, tki, tkv


def segment_counts(d, scratch):
    """Candidates per row of the last row block of a precision-2 long call: the 1,024-byte header, wr_eval_rank_tc's
    layout (A, B, row_ok, anorm, counters, the rank candidate list), then LongScratch (bounds, counts, segments)."""
    rb = max(256, int(16e9 / N_ITEMS) // 256 * 256)
    cap = min(max(int(rb * N_ITEMS / 128.0), 1 << 20), 1 << 27)
    rb = min(rb, LONG_ROWS)
    a_cols = 2 * d if d >= 256 else 3 * d
    off = align(R * a_cols * 2) + align(N_ITEMS * 3 * d * 2) + align(R) + align(R * 4) + 1024
    cnt_at = 1024 + align(off + cap * 8) + align(rb * RANGES * 4)
    last_rows = R - (R - 1) // rb * rb
    return scratch[cnt_at:cnt_at + 4 * last_rows].view(torch.int32)


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
    out = {'what': 'full-ranking eval with top-k lists up to 256, %d rows x %d items, %d-item histories'
                   % (R, N_ITEMS, HIST),
           'gpu': smi, 'reps': a.reps,
           'timing': 'CUDA events per call, median of reps after one warm-up call per shape; precision 0 on the first '
                     '%d rows, scaled per row' % SLICE}
    for d in (64, 128, 256):
        tabs = tables(d, dev)
        U, I, user, pos, hp, hi = tabs
        slice_tabs = (U, I, user[sl].contiguous(), pos[sl].contiguous(), hp, hi)
        n2 = _lib.load().wr_eval_scratch_bytes_topk_long(R, N_ITEMS, d, 2, 256)
        n32 = _lib.load().wr_eval_scratch_bytes_topk(R, N_ITEMS, d, 2, 32)
        n0 = _lib.load().wr_eval_scratch_bytes_topk_long(SLICE, N_ITEMS, d, 0, 256)
        s2, s32, s0 = (_lib._aligned_scratch(n, dev) for n in (n2, n32, n0))
        for k in (32, 64, 100, 256):
            fns = {
                'p2_topk': (lambda: exact_topk_call(tabs, ws, s32, k)) if k <= 32 else
                           (lambda: long_call(tabs, ws, s2, k, 2)),
                'p2_ranks': lambda: _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, precision=2),
                'p0_topk_slice': (lambda: _lib.eval_rank_topk(*slice_tabs, ws, k=k, precision=0)[:4]) if k <= 32 else
                                 (lambda: long_call(slice_tabs, ws, s0, k, 0)),
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
            s2[:4].zero_()
            r2, t2, i2, v2 = fns['p2_topk']()
            rec = {}
            if k > 32:
                cnt = segment_counts(d, s2).to(torch.int64)
                torch.cuda.synchronize()
                rec = {'candidates_per_row_last_block_mean': float(cnt.float().mean()),
                       'candidates_per_row_last_block_max': int(cnt.max()),
                       'candidates_per_row_last_block_p99': float(torch.quantile(cnt.float(), 0.99)),
                       'segment_capacity': 4096, 'fallback_rows': int(s2[:4].view(torch.int32).item())}
            st |= ws.status()
            r0, _, i0, v0 = fns['p0_topk_slice']()
            ranks_only = _lib.eval_rank_topk(U, I, user, pos, hp, hi, ws, precision=2)[0]
            st |= ws.status()
            per_row_p0 = med['p0_topk_slice'] / SLICE
            key = 'd%d_k%d' % (d, k)
            out[key] = dict(
                path='wr_eval_rank_topk (k <= 32)' if k <= 32 else 'wr_eval_rank_topk_long',
                p2_topk_ms=med['p2_topk'], p2_ranks_ms=med['p2_ranks'], p0_topk_slice_ms=med['p0_topk_slice'],
                p0_topk_ms_scaled_to_all_rows=per_row_p0 * R,
                p2_topk_speedup_over_p0_topk_per_row=per_row_p0 / (med['p2_topk'] / R),
                p2_topk_over_p2_ranks=med['p2_topk'] / med['p2_ranks'],
                status=st,
                p2_lists_equal_p0_on_slice=bool(torch.equal(i2[sl], i0) and torch.equal(v2[sl], v0)),
                p2_ranks_equal_p0_on_slice=bool(torch.equal(r2[sl], r0)),
                p2_ranks_equal_ranks_only_call=bool(torch.equal(r2, ranks_only)),
                all_ms=times, **rec)
            if k > 32:
                out[key]['p2_topk_over_p2_k32'] = med['p2_topk'] / out['d%d_k32' % d]['p2_topk_ms']
            print(json.dumps({key: out[key]}), flush=True)
        del tabs, slice_tabs, U, I, s2, s32, s0
        torch.cuda.empty_cache()
    line = json.dumps(out)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, 'bench_eval_topk_long.json'), 'w') as f:
        f.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
