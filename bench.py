#!/usr/bin/env python
"""bench.py -- train interactions/s of the BPRMF hot path (BASELINE.json configs[1]) on N B200s.

    python bench.py --gpus 1 --steps 200 --warmup 10          # this repository's sm_100a path
    python bench.py --impl reference --steps 20 --warmup 3    # the reference's CPU path (oracle port) on host cores
    torchrun --nproc-per-node N bench.py --gpus N ...         # one rank per GPU, tables row-sharded over NVLink

Workload (config.workload): BPRMF, embedding 64, batch 2048, Adam lr=1e-3 l2=1e-6 on the ml-1m-SHAPED synthetic
corpus (6,040 users x 3,706 items, 836k interactions after the reader's rating filter, 668,862 train rows):
`ml-1m.inter` is missing from the reference checkout and there is no network (SURVEY.md fact 3).
A step = one mini-batch through the whole training path (gather + BPR loss + backward scatter + dense Adam/L2 sweep
over every table row): ONE cooperative launch, wr_bprmf_step (wr_bprmf_step_sharded per rank for N > 1, with 2048
rows per GPU and the cross-GPU synchronisation inside the kernel).

value    : interactions/s with the epoch's batches already resident in HBM, device-timed (CUDA events around every
           step, L2 flushed between steps by writing a 512 MB buffer, outside the events), max over ranks.  One
           cooperative launch per step (wr_bprmf_step).
--dump-outputs DIR: after the timed steps, the loss of the last timed step and the user / item embedding tables it left
           (what a caller of train_step receives) are written as DIR/<name>.npy in float32.  The corpus, the initial
           tables and the batches are seeded, so two builds run with the same arguments can be compared array by array.
e2e      : the same through the reference-facing API with HOST batches -- model.train_step_host -> wr_bprmf_ctx_step:
           every step's ids start in ORDINARY (pageable) host memory, are collated into the context's pinned ring, pulled
           over PCIe by the resident training kernel, and the batch loss comes back through mapped host memory; the call
           returns when the whole step is complete.  Host-timed, L2 flushed between steps.  `e2e.pipelined` is the same
           loop with the host running up to 12 steps ahead (what a training loop does; no flush is possible there).
roofline : the step kernel's algorithmic bytes (SURVEY.md 8d: 24 B D + 24 B + 32 D (U + I)) over its event-timed
           duration against the measured HBM copy peak (`frac`), and the same with the DRAM bytes ncu counted for that
           kernel (`achieved_dram`, `traffic`: looked up in profiles/r02_kernel_traffic.json, null when absent).
           `resident_epoch` is the epoch-level form (one launch for 327 steps; tables L2-resident by construction).
extra    : epoch-level fit, eval (fp32 / tcgen05), LightGCN step, the HBM-bound 10M x 2M shape, the reference's step as
           torch CUDA eager ops on the same B200; multi-GPU extras incl. a sharded-vs-single-GPU parity check.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B, D, LR, L2 = 2048, 64, 1e-3, 1e-6
CACHE = os.environ.get('WR_CACHE', os.path.join(tempfile.gettempdir(), 'wr_cache_%d' % os.getuid()))   # one per user
TRAFFIC_FILE = os.path.join(ROOT, 'profiles', 'r02_kernel_traffic.json')   # ncu --set full: dram bytes per launch, by kernel + shape


def measured_traffic(key):
    """{'dram_read', 'dram_write', 'duration_us', 'source'} of one launch of `key` from the committed ncu summary."""
    try:
        return json.load(open(TRAFFIC_FILE)).get(key)
    except (OSError, ValueError):
        return None


WORKLOAD = 'BPRMF emb=64 B=2048 Adam(lr=1e-3,l2=1e-6) on ml-1m-shaped synthetic (6040 users x 3706 items, 668862 train rows)'


_STDOUT_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout: anything a library prints there (NCCL's version banner, torchrun
    notices) is sent to stderr instead; emit() writes the line to the real stdout."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + '\n').encode()
    if _STDOUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_STDOUT_FD, data)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array of `arrays` (name -> tensor) as <out_dir>/<name>.npy in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.asarray(a.detach().cpu().numpy(), dtype=np.float32))


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return p['hbm_gbs'], p.get('bf16_tflops_sustained', 1387.5), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 1590.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.rows.extend(self.proc.stdout.readlines()), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.rows:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


def make_model(corpus, dev, cls_name='BPRMF', **over):
    from whisprrec_b200.main import default_args as model_args
    from whisprrec_b200.models.general.BPRMF import BPRMF
    from whisprrec_b200.models.general.LightGCN import LightGCN
    from whisprrec_b200.helpers.BaseRunner import BaseRunner
    from whisprrec_b200.utils import utils
    cls = {'BPRMF': BPRMF, 'LightGCN': LightGCN}[cls_name]
    args = model_args(cls, lr=LR, l2=L2, batch_size=B, embedding_size=D, **over)
    utils.init_seed(3407)
    model = cls(args, corpus).to(dev)
    model.fuse()
    runner = BaseRunner(args)
    model.optimizer = runner._build_optimizer(model)
    data = {ph: cls.Dataset(model, corpus, ph) for ph in ('train', 'dev')}
    return model, runner, data


def algorithmic_bytes_adam(n_rows, d):
    return 32 * d * n_rows            # read p, m, v, g; write p, m, v, g=0 (SURVEY.md section 8d)


def algorithmic_bytes_bpr(b, d):
    return 24 * b * d + 24 * b        # 3 gathered rows + 3 gradient rows of 4D bytes, 3 int64 ids


def roofline_block(step_bytes, step_avg_s, hbm_peak, peak_src, ep_us_per_step):
    achieved = step_bytes / step_avg_s / 1e9
    tr = measured_traffic('bprmf_step_kernel<16,1,LocalTabs>@ml1m_b2048_flushed')
    traffic = None if tr is None else tr['dram_read'] + tr['dram_write']
    out = {'bound': 'hbm', 'kernel': 'bprmf_step_kernel<16,1,LocalTabs>', 'achieved': achieved, 'peak': hbm_peak,
           'unit': 'GB/s', 'frac': achieved / hbm_peak, 'traffic': traffic,
           'achieved_dram': None if traffic is None else traffic / step_avg_s / 1e9,
           'frac_dram': None if traffic is None else traffic / step_avg_s / 1e9 / hbm_peak,
           'traffic_source': None if tr is None else tr.get('source'),
           'peak_source': peak_src, 'bytes_per_launch': step_bytes, 'avg_launch_us': step_avg_s * 1e6,
           'note': 'one launch per step with a cold L2: a latency chain (ids -> rows -> REDs -> grid barrier -> Adam) on 23 MB, '
                   'of which ~8 us is the launch/event floor (scripts/prof_resident.py); the same arithmetic where HBM is '
                   'the bound: extra.bprmf_10Mx2M_d128_b65536',
           'resident_epoch': {'kernel': 'bprmf_epoch_owner_kernel<8,2> (one grid barrier per step; WR_EPOCH_KERNEL=two_barrier: '
                                        'bprmf_epoch_kernel<16,1>)', 'us_per_step': ep_us_per_step,
                              'achieved': step_bytes / (ep_us_per_step * 1e-6) / 1e9,
                              'frac': step_bytes / (ep_us_per_step * 1e-6) / 1e9 / hbm_peak,
                              'note': 'ALGORITHMIC bytes over the per-step time of the one-launch epoch; the tables stay in '
                                      'L2 / shared memory between steps (that is the design), so this is not a DRAM rate'}}
    return out


def torch_eager_b200(corpus, dev, batches, n_steps=60):
    """SURVEY.md 8d(ii): the reference's own step as torch CUDA eager ops on this B200 -- nn.Embedding gathers, the row
    dots, BPRLoss (utils/loss.py:33-39), autograd, torch.optim.Adam(weight_decay) (BaseRunner.py:120-124,196-199) --
    i.e. what `main.py --gpu 0` executes per batch, on the same batches, model-only (no DataLoader)."""
    import torch.nn as nn
    torch.manual_seed(3407)
    ue, ie = nn.Embedding(corpus.n_users, D).to(dev), nn.Embedding(corpus.n_items, D).to(dev)
    opt = torch.optim.Adam(list(ue.parameters()) + list(ie.parameters()), lr=LR, weight_decay=L2)
    spe = batches.shape[1] // B

    def step(s):
        lo = (s % spe) * B
        u, p, n = batches[0, lo:lo + B], batches[1, lo:lo + B], batches[2, lo:lo + B]
        opt.zero_grad()
        uu = ue(u)
        sp, sn = (uu * ie(p)).sum(-1), (uu * ie(n)).sum(-1)
        loss = -torch.log(1e-10 + torch.sigmoid(sp - sn)).mean()
        loss.backward()
        opt.step()
        return loss
    for s in range(10):
        step(s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for s in range(n_steps):
        loss = step(10 + s)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    lh = float(loss)
    return {'interactions_per_s': n_steps * B / wall, 'ms_per_step_wall': wall / n_steps * 1e3,
            'ms_per_step_device': e0.elapsed_time(e1) / n_steps, 'steps': n_steps, 'loss_finite': bool(np.isfinite(lh)),
            'how': 'torch %s CUDA eager, fp32, back-to-back steps without a per-step sync (the reference syncs every step: '
                   'BaseRunner.py:200), tables L2-resident' % torch.__version__}


def run_ours(a, rank, world, local_rank):
    from whisprrec_b200.utils import synthetic
    from whisprrec_b200 import _lib as _lib_mod
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    hbm_peak, _, peak_src = peaks()
    corpus = synthetic.ml1m_shaped_corpus(cache_dir=os.path.join(CACHE, 'r%d' % rank))
    model, runner, data = make_model(corpus, dev)
    t = model.tables
    n_rows = t.P.shape[0]
    batches = runner.epoch_batches(data['train'])              # [3, n_train] int64, resident
    n_train = batches.shape[1]
    steps_per_epoch = n_train // B                             # full batches only inside the timed region
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    losses = torch.zeros(a.warmup + a.steps, device=dev)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(a.steps)]

    def step(s, events=None):
        lo = (s % steps_per_epoch) * B
        batch = {'user_id': batches[0, lo:lo + B], 'pos_item': batches[1, lo:lo + B], 'neg_items': batches[2, lo:lo + B]}
        if events: events[0].record()
        model.train_step(batch, loss_out=losses[s:s + 1])     # what BaseRunner.fit calls: one cooperative launch
        if events: events[1].record()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            torch.cuda.synchronize()

    for s in range(a.warmup):
        flush.zero_()
        step(s)
    barrier()
    with ClockSampler(local_rank) as clk:
        wall0 = time.perf_counter()
        for s in range(a.steps):
            flush.zero_()                                      # L2 flush, outside the per-step events
            step(a.warmup + s, ev[s])
        barrier()
        wall = time.perf_counter() - wall0
        if a.dump_outputs:                                     # before the untimed steps below
            last = {'loss': losses[a.warmup + a.steps - 1:].cpu(), 'user_embeddings': t.users(t.P).cpu(),
                    'item_embeddings': t.items(t.P).cpu()}
        if wall < 1.5:                                         # keep the sampler alive long enough to see clocks
            t_end = time.perf_counter() + 1.5 - wall
            while time.perf_counter() < t_end:
                flush.zero_(); step(0)
            torch.cuda.synchronize()
    clocks = clk.summary()
    step_ms = np.array([e[0].elapsed_time(e[1]) for e in ev])
    total_ms = float(step_ms.sum())
    if world > 1:
        import torch.distributed as dist
        tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt.item())
    t.ws.raise_on_status()
    assert np.isfinite(losses.cpu().numpy()).all()
    value = world * a.steps * B / (total_ms * 1e-3)

    # ---- e2e: every step's ids start in pageable host memory; collate -> pinned ring -> PCIe -> step -> loss on the host ----
    host_batches = batches.cpu()
    n_buf = min(steps_per_epoch, 64)
    pageable = [host_batches[:, s * B:(s + 1) * B].contiguous() for s in range(n_buf)]      # what collate_batch hands over
    pinned = [t_.pin_memory() for t_ in pageable]
    cur = torch.cuda.current_stream()

    def e2e_loop(bufs, n_warm, n_timed, do_flush):
        tot = 0.0
        for s in range(n_warm + n_timed):
            if do_flush:
                flush.zero_()
                cur.synchronize()        # the flush only: the resident training kernel lives on its own stream
            t0 = time.perf_counter()
            loss = model.train_step_host(bufs[s % n_buf])       # returns when the whole step is complete
            if s >= n_warm:
                tot += time.perf_counter() - t0
        return tot, loss
    e2e_s, loss_host = e2e_loop(pageable, max(a.warmup, 10), a.steps, True)
    e2e_pinned_s, _ = e2e_loop(pinned, 5, a.steps, True)
    e2e_warm_s, _ = e2e_loop(pageable, 5, a.steps, False)
    # the host running ahead (a training loop): push without waiting, collect the loss 12 steps later
    n_pipe = max(a.steps, 400)
    model.quiesce()
    k0 = model._host_ctx.steps
    t0 = time.perf_counter()
    for s in range(n_pipe):
        model.train_step_host(pageable[s % n_buf], wait=0)
        if s >= 12:
            loss_pipe = model.host_step_loss(k0 + s - 12)
    for s in range(n_pipe - 12, n_pipe):
        loss_pipe = model.host_step_loss(k0 + s)
    e2e_pipe_s = time.perf_counter() - t0
    model.quiesce()
    torch.cuda.synchronize()
    # the copy-engine form with a stream synchronisation per step (wr_bprmf_step_host), for comparison
    t = model.tables
    stage, pl = torch.empty(3 * B, dtype=torch.int64, device=dev), torch.zeros(1).pin_memory()
    e2e_copy_s = 0.0
    for s in range(a.warmup + a.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.optimizer.step_count += 1
        _lib_mod.bprmf_step_host(pinned[s % n_buf], stage, pl, t.P, t.M, t.V, t.G, t.n_users,
                                 model.optimizer.step_count, LR, L2, t.loss, t.ws)
        loss_host2 = float(pl[0])
        if s >= a.warmup:
            e2e_copy_s += time.perf_counter() - t0
    assert np.isfinite(loss_host) and np.isfinite(loss_pipe) and np.isfinite(loss_host2)
    t.ws.raise_on_status()
    e2e_value = world * a.steps * B / e2e_s

    # ---- the epoch-level form of the same steps: ONE resident launch for all 327 (what BaseRunner.fit calls) ----
    ep_losses = torch.zeros(steps_per_epoch + 1, device=dev)
    ids_epoch = batches[:, :steps_per_epoch * B].contiguous()
    ep_ms = []
    for r in range(7):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        model.train_epoch(ids_epoch, B, ep_losses)
        e1.record()
        torch.cuda.synchronize()
        ep_ms.append(e0.elapsed_time(e1))
    assert np.isfinite(ep_losses[:steps_per_epoch].cpu().numpy()).all()
    ep_us_per_step = float(np.median(ep_ms[2:])) * 1e3 / steps_per_epoch

    step_bytes = algorithmic_bytes_adam(n_rows, D) + algorithmic_bytes_bpr(B, D)
    step_avg_s = float(step_ms.mean()) * 1e-3
    achieved = step_bytes / step_avg_s / 1e9
    line = {
        'metric': 'train_interactions_per_s', 'value': value, 'unit': 'interactions/s', 'n_gpus': world,
        'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': total_ms / a.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'batch_per_gpu': B, 'embedding_size': D, 'table_rows': int(n_rows),
                   'l2_flush': '512 MB written between timed steps (tables are 10 MB, L2-resident otherwise)',
                   'parallelism': 'single GPU' if world == 1 else 'replicas x%d' % world},
        'e2e': {'value': e2e_value, 'unit': 'interactions/s', 'h2d_bytes_per_step': 3 * B * 8,
                'd2h_bytes_per_step': 12, 'ms_per_step': e2e_s / a.steps * 1e3,
                'how': 'model.train_step_host -> wr_bprmf_ctx_step on the resident kernel: ids start in PAGEABLE host '
                       'memory (collated into the pinned ring inside the call), are pulled over PCIe by the kernel\'s helper '
                       'warps, loss + completion words come back through mapped host memory; every call returns when its '
                       'step is complete; L2 flushed (512 MB) before every step, outside the timer',
                'pinned_in_place': {'value': world * a.steps * B / e2e_pinned_s, 'ms_per_step': e2e_pinned_s / a.steps * 1e3,
                                    'how': 'the same with the ids already in pinned memory (read in place, no collate copy)'},
                'no_flush': {'value': world * a.steps * B / e2e_warm_s, 'ms_per_step': e2e_warm_s / a.steps * 1e3,
                             'how': 'pageable ids, every step waited for, tables L2-resident (no flush)'},
                'pipelined': {'value': world * n_pipe * B / e2e_pipe_s, 'ms_per_step': e2e_pipe_s / n_pipe * 1e3, 'steps': n_pipe,
                              'how': 'pageable ids, wait=0: the host runs up to 12 steps ahead and reads every loss 12 steps '
                                     'later (a training loop); no flush is possible between pipelined steps'},
                'copy_engine_form': {'value': world * a.steps * B / e2e_copy_s, 'ms_per_step': e2e_copy_s / a.steps * 1e3,
                                     'how': 'wr_bprmf_step_host: cudaMemcpyAsync H2D + step + cudaMemcpyAsync D2H + '
                                            'cudaStreamSynchronize'}},
        'gpu_launches': a.steps,
        'clocks': clocks,
        'roofline': roofline_block(step_bytes, step_avg_s, hbm_peak, peak_src, ep_us_per_step),
        'kernels_ms': {'bprmf_step': float(step_ms.mean()), 'step_median': float(np.median(step_ms))},
    }
    if rank == 0 and world == 1:
        line['cpu_baseline'] = cpu_baseline(corpus, budget_s=a.cpu_budget)
        if not a.no_extras:
            line['extra'] = extras(corpus, dev, model, runner, data, hbm_peak)
            try:
                line['extra']['torch_eager_b200'] = torch_eager_b200(corpus, dev, batches)
            except Exception as e:  # noqa: BLE001
                line['extra']['torch_eager_b200'] = {'error': repr(e)}
    if rank == 0:
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, last)
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def run_ours_sharded(a, rank, world, local_rank):
    """N > 1: the same tables row-sharded over the N GPUs (NVLink peer memory, whisprrec_b200/sharded.py); every
    step trains one GLOBAL batch of N x 2048 interactions, each rank feeding its 2048-row slice (weak scaling)."""
    import torch.distributed as dist
    from whisprrec_b200 import _lib, sharded as S
    from whisprrec_b200.utils import synthetic
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    hbm_peak, _, peak_src = peaks()
    corpus = synthetic.ml1m_shaped_corpus(cache_dir=os.path.join(CACHE, 'r%d' % rank))
    model, runner, data = make_model(corpus, dev)
    peers = S.PeerGroup(dev)
    st = model.shard(peers)
    batches = runner.epoch_batches(data['train'])              # identical on every rank (same seeds)
    GB = B * world
    steps_per_epoch = batches.shape[1] // GB
    lo_r = rank * B                                            # this rank's slice of every global batch
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    losses = torch.zeros(a.warmup + a.steps, device=dev)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(a.steps)]

    def step(s, events=None):
        lo = (s % steps_per_epoch) * GB + lo_r
        u, p, n = batches[0, lo:lo + B], batches[1, lo:lo + B], batches[2, lo:lo + B]
        if events: events[0].record()
        loss = model.sharded_train_step(u, p, n, GB, LR, L2)      # one cooperative launch per rank (wr_bprmf_step_sharded)
        if events: events[1].record()
        losses[s:s + 1].copy_(loss[:1])

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    parity = sharded_parity(model, runner, data, st, peers, batches, GB, lo_r, dev)
    for s in range(a.warmup):
        flush.zero_()
        step(s)
    barrier()
    with ClockSampler(local_rank) as clk:
        wall0 = time.perf_counter()
        for s in range(a.steps):
            flush.zero_()
            step(a.warmup + s, ev[s])
        barrier()
        wall = time.perf_counter() - wall0
        if a.dump_outputs:                                     # before the untimed steps below; every rank takes part
            gu, gi = st.gather_full()
            last = {'loss': losses[a.warmup + a.steps - 1:].cpu(), 'user_embeddings': gu.cpu(), 'item_embeddings': gi.cpu()}
        extra_steps = int(max(0.0, 1.5 - wall) / 2e-4) if wall < 1.5 else 0
        t_extra = torch.tensor([extra_steps], device=dev)
        dist.all_reduce(t_extra, op=dist.ReduceOp.MAX)         # every rank runs the same number of steps
        for s in range(int(t_extra.item())):
            flush.zero_(); step(0)
        barrier()
    clocks = clk.summary()
    step_ms = np.array([e[0].elapsed_time(e[1]) for e in ev])
    tt = torch.tensor([float(step_ms.sum())], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    st.ws.raise_on_status()
    assert np.isfinite(losses.cpu().numpy()).all()
    value = a.steps * GB / (total_ms * 1e-3)

    # ---- e2e: each rank's slice comes from pinned host memory every step, the loss goes back to the host ----
    host_batches = batches.cpu()
    pinned = torch.empty((steps_per_epoch, 3, B), dtype=torch.int64).pin_memory()
    for s in range(steps_per_epoch):
        pinned[s].copy_(host_batches[:, s * GB + lo_r:s * GB + lo_r + B])
    stage = torch.empty((3, B), dtype=torch.int64, device=dev)
    e2e_s = 0.0
    for s in range(a.warmup + a.steps):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        stage.copy_(pinned[s % steps_per_epoch], non_blocking=True)
        loss = model.sharded_train_step(stage[0], stage[1], stage[2], GB, LR, L2)
        loss_host = float(loss[0])
        if s >= a.warmup:
            e2e_s += time.perf_counter() - t0
    tt = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_s = float(tt.item())
    assert np.isfinite(loss_host)

    n_local = st.layout.n_local
    step_bytes = algorithmic_bytes_adam(n_local, D) + algorithmic_bytes_bpr(B, D)          # per GPU
    step_avg_s = float(step_ms.mean()) * 1e-3
    # the multi-launch form of the same step (what shards too large for the single launch use), timed piecewise
    seg_ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(20)]
    for e in seg_ev:
        flush.zero_()
        lo = lo_r
        u, p, n = batches[0, lo:lo + B], batches[1, lo:lo + B], batches[2, lo:lo + B]
        peers.barrier()
        e[0].record()
        _lib.bpr_fwd_bwd_sharded(st.T, st.Gd, u, p, n, GB, st.D, st.loss_part, st.ws)
        e[1].record()
        peers.barrier(st.loss_part[:1])
        e[2].record()
        st.adam(LR, L2)
        e[3].record()
        peers.barrier()
        e[4].record()
    barrier()
    seg = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(4)] for e in seg_ev])
    line = {
        'metric': 'train_interactions_per_s', 'value': value, 'unit': 'interactions/s', 'n_gpus': world,
        'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': total_ms / a.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'batch_per_gpu': B, 'global_batch': GB, 'embedding_size': D,
                   'table_rows': int(st.layout.n_users + st.layout.n_items), 'table_rows_per_gpu': int(n_local),
                   'l2_flush': '512 MB written between timed steps on every GPU',
                   'parallelism': 'tables row-sharded x%d over NVLink peer memory; one cooperative launch per GPU and '
                                  'step: remote gathers and gradient REDs, the cross-GPU barriers and the loss '
                                  'all-reduce all happen inside the kernel (no collective call)' % world},
        'e2e': {'value': a.steps * GB / e2e_s, 'unit': 'interactions/s', 'h2d_bytes_per_step': 3 * B * 8 * world,
                'd2h_bytes_per_step': 4 * world, 'ms_per_step': e2e_s / a.steps * 1e3},
        'gpu_launches': a.steps,
        'clocks': clocks,
        'roofline': {'bound': 'hbm', 'kernel': 'bprmf_step_kernel<ShardTabs>', 'achieved': step_bytes / step_avg_s / 1e9,
                     'peak': hbm_peak, 'unit': 'GB/s', 'frac': step_bytes / step_avg_s / 1e9 / hbm_peak, 'traffic': None,
                     'peak_source': peak_src, 'bytes_per_launch': step_bytes, 'avg_launch_us': step_avg_s * 1e6,
                     'note': 'per GPU; (world-1)/world of the gathered rows and gradient REDs cross NVLink; latency-bound '
                             '(launch + DRAM and NVLink round trips + two cross-GPU meeting points)'},
        'kernels_ms': {'bprmf_step_sharded': float(step_ms.mean()), 'step_median': float(np.median(step_ms)),
                       'multi_launch_form': {'bpr_fwd_bwd_sharded': float(seg[:, 0].mean()),
                                             'barrier_after_scatter': float(seg[:, 1].mean()),
                                             'adam_l2_sweep': float(seg[:, 2].mean()),
                                             'barrier_after_adam': float(seg[:, 3].mean())}},
    }
    line['extra'] = {'parity': parity}
    if not a.no_extras:
        line['extra'].update(extras_sharded(peers, dev, hbm_peak, flush))
    if rank == 0:
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, last)
        emit(line)
    peers.close()
    dist.destroy_process_group()


def sharded_parity(model, runner, data, st, peers, batches, GB, lo_r, dev):
    """Before anything is timed: three global batches through the sharded step on the N GPUs and through the single-GPU
    step on this rank's full replica of the tables (still in place from before model.shard()), then the sharded
    full-ranking evaluation of the dev split against the single-GPU kernel on the gathered tables.  Asserted on every
    rank (a failure aborts the bench) and reported under extra.parity."""
    import torch.distributed as dist
    from whisprrec_b200 import _lib
    t = model.tables
    Pf, Mf, Vf, Gf = t.P.clone(), t.M.clone(), t.V.clone(), t.G.clone()
    lossf = torch.zeros(1, device=dev)
    worst_loss, worst_p = 0.0, 0.0
    for k in range(3):
        lo = k * GB
        u, p, n = batches[0, lo:lo + GB], batches[1, lo:lo + GB], batches[2, lo:lo + GB]
        loss = model.sharded_train_step(u[lo_r:lo_r + B].contiguous(), p[lo_r:lo_r + B].contiguous(),
                                        n[lo_r:lo_r + B].contiguous(), GB, LR, L2)
        _lib.bpr_fwd_bwd(Pf[:t.n_users], Pf[t.n_users:], u.contiguous(), p.contiguous(), n.contiguous(),
                         Gf[:t.n_users], Gf[t.n_users:], lossf, t.ws)
        _lib.adam_l2_sweep(Pf, Mf, Vf, Gf, st.step_count, LR, L2)
        a_, b_ = float(loss[0]), float(lossf[0])
        worst_loss = max(worst_loss, abs(a_ - b_) / abs(b_))
        gu, gi = st.gather_full()
        full = torch.cat([gu, gi])
        err = ((full - Pf).abs() - 1e-5 * Pf.abs()).max().item() / float(Pf.abs().max())
        worst_p = max(worst_p, err)
        peers.barrier()
    assert worst_loss <= 2e-6, ('sharded loss differs from the single-GPU step', worst_loss)
    assert worst_p <= 2e-6, ('sharded parameters differ from the single-GPU step', worst_p)
    # evaluation: item-sharded ranks against the single-GPU kernel on the same (gathered) tables -- identical
    (user, pos), (hptr, hidx) = runner._eval_inputs(data['dev'])
    got = runner.rank_topk(data['dev'])[0]
    gu, gi = st.gather_full()
    want = _lib.eval_rank_topk(gu.contiguous(), gi.contiguous(), user, pos, hptr, hidx, t.ws)[0]
    mism = int((got != want).sum().item())
    assert mism == 0, ('sharded eval ranks differ from the single-GPU kernel', mism)
    ok = torch.tensor([1], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    st.ws.raise_on_status()
    return {'ok': bool(ok.item()), 'steps': 3, 'loss_rel_err_max': worst_loss, 'loss_bound': 2e-6,
            'param_excess_over_1e-5_rel_max': worst_p, 'param_bound': '|a-b| <= 1e-5 |b| + 2e-6 max|b|',
            'eval_rows': int(user.numel()), 'eval_rank_mismatches': mism,
            'against': 'wr_bpr_fwd_bwd + wr_adam_l2_sweep and wr_eval_rank_topk on one GPU, same batches'}


def extras_sharded(peers, dev, hbm_peak, flush):
    """Secondary multi-GPU measurements: the HBM-bound BPRMF shape (10M x 2M, D=128) with the tables row-sharded, and
    item-sharded tensor-core evaluation.  Every rank runs them; the numbers are rank 0's device times (max over ranks)."""
    import torch.distributed as dist
    from whisprrec_b200 import _lib, sharded as S
    out = {}
    world, rank = peers.world, peers.rank

    def timed_max(fn, reps):
        ms = []
        for _ in range(reps):
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        t = torch.tensor([float(np.median(ms))], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    try:
        nU, nI, d, b = 10_000_000, 2_000_000, 128, 65536
        lay = S.ShardLayout(nU, nI, world, rank)
        tabs = S.ShardedTables(peers, lay, d)
        tabs.P.normal_(0, 0.01)
        peers.host_sync()
        g = torch.Generator(device=dev); g.manual_seed(100 + rank)
        u = torch.randint(0, nU, (b,), device=dev, generator=g)
        p = torch.randint(0, nI, (b,), device=dev, generator=g)
        n = torch.randint(1, nI, (b,), device=dev, generator=g)
        step = lambda: S.bprmf_step(tabs, u, p, n, b * world, LR, L2)
        step()
        ms = timed_max(step, 5)
        # the row-marked sweep moves 24 B per parameter (G is read and re-zeroed only in the rows that received a gradient)
        step_bytes = algorithmic_bytes_adam(lay.n_local, d) * 3 // 4 + algorithmic_bytes_bpr(b, d)
        out['bprmf_10Mx2M_d128_b65536_per_gpu_sharded'] = {
            'ms_per_step': ms, 'interactions_per_s': b * world / (ms * 1e-3), 'rows_per_gpu': lay.n_local,
            'algorithmic_gbs_per_gpu': step_bytes / (ms * 1e-3) / 1e9,
            'frac_of_hbm_peak': step_bytes / (ms * 1e-3) / 1e9 / hbm_peak,
            'note': 'total table fixed (24.6 GB of state over all GPUs), batch 65536 per GPU; row exchange (request lists to '
                    'the owners, owners store the rows into the requesters\' buffers, batch kernel on local memory, gradient '
                    'rows into the owners\' inboxes: posted NVLink stores only), local inbox reduction, row-marked local Adam '
                    'sweep (24 B per parameter); 3 cross-GPU barriers per step'}
        del tabs
    except Exception as e:  # noqa: BLE001
        out['bprmf_10Mx2M_d128_b65536_per_gpu_sharded'] = {'error': repr(e)}
    try:    # BASELINE.json configs[3]: LightGCN L=3 D=128, 10M x 2M x 494M edges, rows sharded over the N GPUs
        import argparse as _ap
        from scripts.bench_lightgcn_scale import run as lightgcn_scale
        torch.cuda.empty_cache()
        cfg = _ap.Namespace(users=10_000_000, items=2_000_000, edges=500_000_000, dim=128, layers=3, batch=65536, steps=3, warmup=1)
        out['lightgcn_cfg4_10Mx2Mx494M_L3_d128_sharded'] = lightgcn_scale(cfg, rank, world, dev, peers)
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out['lightgcn_cfg4_10Mx2Mx494M_L3_d128_sharded'] = {'error': repr(e)}
    try:
        _, tensor_peak, _ = peaks()
        for d in (64, 128):
            nUs, nIs, Rs = 200_000, 1_000_000, 262_144
            lay = S.ShardLayout(nUs, nIs, world, rank)
            tabs = S.ShardedTables(peers, lay, d)
            g = torch.Generator(device=dev); g.manual_seed(3407 + rank)
            tabs.P.copy_(torch.randn((lay.n_local, d), device=dev, generator=g) / d ** 0.5)
            peers.host_sync()
            g2 = torch.Generator(device=dev); g2.manual_seed(3407)
            us = torch.randint(0, nUs, (Rs,), device=dev, generator=g2)
            ps = torch.randint(0, nIs, (Rs,), device=dev, generator=g2)
            hl = 50 // world + 1
            hp_ = torch.arange(0, (nUs + 1) * hl, hl, device=dev, dtype=torch.int64)
            n_loc_items = len(lay.local_items())
            hi_ = torch.sort(torch.randint(0, n_loc_items, (nUs, hl), device=dev, generator=g2), dim=1).values \
                .to(torch.int32).reshape(-1).contiguous()
            fn = lambda: S.sharded_eval(tabs, tabs.T, tabs.item_rows(tabs.P), us, ps, (hp_, hi_), precision=1)
            fn()
            ms = timed_max(fn, 3)
            tf = 2.0 * Rs * nIs * d / (ms * 1e-3) / 1e12
            out['eval_tcgen05_item_sharded_262144x1M_d%d' % d] = {
                'users_per_s': Rs / (ms * 1e-3), 'ms': ms, 'job_tflops': tf, 'tflops_per_gpu': tf / world,
                'frac_of_bf16_peak_per_gpu': tf / world / tensor_peak}
            del tabs
    except Exception as e:  # noqa: BLE001
        out['eval_tcgen05_item_sharded'] = {'error': repr(e)}
    return out


def cpu_problem(corpus):
    """The same workload for the CPU arm: reference-initialised tables and one epoch of reference-ordered batches."""
    from whisprrec_b200.main import default_args as model_args
    from whisprrec_b200.models.general.BPRMF import BPRMF
    from whisprrec_b200.helpers.BaseRunner import dataloader_draws
    from whisprrec_b200.utils import utils
    args = model_args(BPRMF, lr=LR, l2=L2, batch_size=B, embedding_size=D)
    args.device = torch.device('cpu')
    utils.init_seed(3407)
    model = BPRMF(args, corpus)
    ds = BPRMF.Dataset(model, corpus, 'train')
    ds.actions_before_epoch()
    perm = dataloader_draws(len(ds), shuffle=True)
    cols = [np.asarray(ds.data[k], dtype=np.int64)[perm] for k in ('user_id', 'item_id', 'neg_items')]
    return model.user_embeddings.weight.detach().clone(), model.item_embeddings.weight.detach().clone(), cols


def cpu_steps(U, I, cols, n_steps, start=0):
    """n_steps of the oracle's restatement of predict -> backward -> Adam.step (reference BaseRunner.py:196-199)."""
    from oracle import whispr_oracle as O
    st = getattr(cpu_steps, 'state', None)
    if st is None or st[0] is not U:
        st = cpu_steps.state = (U, [torch.zeros_like(U), torch.zeros_like(U), torch.zeros_like(I), torch.zeros_like(I)], [0])
    mU, vU, mI, vI = st[1]
    spe = len(cols[0]) // B
    t0 = time.perf_counter()
    for s in range(start, start + n_steps):
        lo = (s % spe) * B
        loss, gU, gI = O.bpr_fwd_bwd(U, I, cols[0][lo:lo + B], cols[1][lo:lo + B], cols[2][lo:lo + B])
        st[2][0] += 1
        O.adam_l2_step(U, mU, vU, gU, st[2][0], LR, L2)
        O.adam_l2_step(I, mI, vI, gI, st[2][0], LR, L2)
    return time.perf_counter() - t0, float(loss)


def cpu_baseline(corpus, budget_s=12.0):
    U, I, cols = cpu_problem(corpus)
    t3, _ = cpu_steps(U, I, cols, 3)
    n = int(max(5, min(3000, budget_s / max(t3 / 3, 1e-6))))
    dt, loss = cpu_steps(U, I, cols, n, start=3)
    return {'value': n * B / dt, 'unit': 'interactions/s', 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': '%d steps of B=%d of the same workload through oracle/whispr_oracle.py (torch CPU ops, '
                      'model-only: batches pre-assembled); host has %d logical cores' % (n, B, os.cpu_count())}


def run_reference(a, rank):
    """The reference arm: the reference's CPU implementation of the path.  The reference is pure Python on top of
    torch and cannot travel to the GPU box, so this is the oracle port of it, on all host threads."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers: this arm must use the host's cores whatever launched it
    torch.set_num_threads(os.cpu_count() or 1)
    from whisprrec_b200.utils import synthetic
    corpus = synthetic.ml1m_shaped_corpus(cache_dir=os.path.join(CACHE, 'ref'))
    U, I, cols = cpu_problem(corpus)
    per_step = 100                                            # a "step" of this arm = a bounded sample of 100 batches
    cpu_steps(U, I, cols, a.warmup * 5)
    dt = 0.0
    for k in range(a.steps):
        d, loss = cpu_steps(U, I, cols, per_step, start=a.warmup * 5 + k * per_step)
        dt += d
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {'loss': torch.tensor([loss]), 'user_embeddings': U, 'item_embeddings': I})
    value = a.steps * per_step * B / dt
    sample = '%d batches of B=%d per step, model-only (batches pre-assembled), oracle port of the reference' % (per_step, B)
    emit({
        'impl': 'reference', 'metric': 'train_interactions_per_s', 'value': value, 'unit': 'interactions/s',
        'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': dt / a.steps * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'batch_per_gpu': B, 'embedding_size': D},
        'cpu_baseline': {'value': value, 'unit': 'interactions/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                         'sample': sample},
        'e2e': {'value': value, 'unit': 'interactions/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    })


# ---------------------------------------------------------------------------------------------------------------
# secondary measurements (reported under "extra"; never replace the contract fields)
# ---------------------------------------------------------------------------------------------------------------

def timed(fn, reps, flush=None):
    ms = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(np.mean(ms))


def extras(corpus, dev, model, runner, data, hbm_peak):
    from whisprrec_b200 import _lib
    from whisprrec_b200.utils import synthetic
    out = {}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    try:    # full-ranking eval of the dev split, fp32-exact kernel
        (user, pos), (hptr, hidx) = runner._eval_inputs(data['dev'])
        ue, ie = model.eval_tables()
        fn = lambda: _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws)
        fn(); torch.cuda.synchronize()
        med, _ = timed(fn, 10, flush)
        R, nI = user.numel(), ie.shape[0]
        out['eval_fp32'] = {'users_per_s': R / (med * 1e-3), 'rows': R, 'items': nI, 'ms': med,
                            'tflops': 2.0 * R * nI * D / (med * 1e-3) / 1e12}
        fn = lambda: _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws, k=10)
        fn(); torch.cuda.synchronize()
        med, _ = timed(fn, 5, flush)
        out['eval_fp32_top10'] = {'users_per_s': R / (med * 1e-3), 'ms': med}
    except Exception as e:  # noqa: BLE001
        out['eval_fp32'] = {'error': repr(e)}
    try:    # whole epochs through BaseRunner.fit: device negative sampling (bit-exact NumPy stream), host permutation,
        #     one step launch per batch, one loss read-back per epoch -- what `main.py` does per epoch
        ep = []
        for _ in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            runner.fit(data['train'])
            torch.cuda.synchronize()
            ep.append((time.perf_counter() - t0, dict(runner.last_epoch_stats)))
        ep.sort(key=lambda x: x[0])
        wall, st = ep[len(ep) // 2]
        out['epoch_fit'] = {'rows': st['rows'], 'steps': st['steps'], 'wall_s': wall, 'host_prep_s': st['host_prep_s'],
                            'device_s': st['device_s'], 'interactions_per_s': st['rows'] / wall,
                            'note': 'sampling + shuffle + upload + all steps + loss read-back; tables L2-resident'}
    except Exception as e:  # noqa: BLE001
        out['epoch_fit'] = {'error': repr(e)}
    try:    # ml-100k (the reference's own CPU-runnable case, BASELINE.json configs[0]): whole epochs and the dev evaluation
        c100 = synthetic.corpus_from_npz(os.path.join(ROOT, 'tests', 'golden', 'ml100k_corpus.npz'))
        res = {}
        for name, over in (('BPRMF', {}), ('LightGCN', {'gcn_layers': 2})):
            m100, r100, d100 = make_model(c100, dev, name, **over)
            r100.fit(d100['train'])
            ep = []
            for _ in range(3):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                r100.fit(d100['train'])
                torch.cuda.synchronize(); ep.append(time.perf_counter() - t0)
            ev = []
            for _ in range(3):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                r100.evaluate(d100['dev'], [10], ['NDCG', 'HR'])
                torch.cuda.synchronize(); ev.append(time.perf_counter() - t0)
            n_tr, n_dev = len(d100['train']), len(d100['dev'])
            res[name] = {'epoch_s': float(np.median(ep)), 'train_interactions_per_s': n_tr / float(np.median(ep)),
                         'dev_eval_s': float(np.median(ev)), 'eval_rows_per_s': n_dev / float(np.median(ev))}
        try:    # SGL (SURVEY.md section 8 f-3): whole epochs incl. the two edge-dropout views per epoch
            from whisprrec_b200.main import default_args as _da
            from whisprrec_b200.models.general.SGL import SGL
            from whisprrec_b200.helpers.BaseRunner import BaseRunner as _BR
            from whisprrec_b200.utils import utils as _u
            sa = _da(SGL, lr=1e-3, l2=0.0, batch_size=B, embedding_size=D)
            _u.init_seed(3407)
            sm = SGL(sa, c100).to(dev)
            sm.fuse()
            sr = _BR(sa)
            sm.optimizer = sr._build_optimizer(sm)
            sd = {ph: SGL.Dataset(sm, c100, ph) for ph in ('train', 'dev')}
            sr.fit(sd['train'])
            ep = []
            for _ in range(3):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                sr.fit(sd['train'])
                torch.cuda.synchronize(); ep.append(time.perf_counter() - t0)
            res['SGL'] = {'epoch_s': float(np.median(ep)), 'train_interactions_per_s': len(sd['train']) / float(np.median(ep)),
                          'note': 'views redrawn every epoch (Python random stream on the host, CSR + transposed CSR on the device); '
                                  'the unmodified reference needs 10.3 s for its first ml-100k epoch on the CPU (DESIGN.md r1 probe)'}
        except Exception as e:  # noqa: BLE001
            res['SGL'] = {'error': repr(e)}
        res['reference_cpu'] = {'note': 'unmodified reference on an 8-core host (BASELINE.md section 2): BPRMF epoch 1.4 s '
                                        '(47k interactions/s), LightGCN 1.7 s (39k/s), dev eval 1.3 s (6.3k rows/s)'}
        out['ml100k'] = res
    except Exception as e:  # noqa: BLE001
        out['ml100k'] = {'error': repr(e)}
    try:    # the two-launch form of the same step (what large tables use): fwd+bwd kernel, then the Adam sweep
        t = model.tables
        batches = runner.epoch_batches(data['train'])
        u, p_, n_ = batches[0, :B].contiguous(), batches[1, :B].contiguous(), batches[2, :B].contiguous()
        bpr = lambda: _lib.bpr_fwd_bwd(t.users(t.P), t.items(t.P), u, p_, n_, t.users(t.G), t.items(t.G), t.loss, t.ws)
        adam = lambda: _lib.adam_l2_sweep(t.P, t.M, t.V, t.G, 1000, LR, L2)
        bmed, _ = timed(bpr, 20, flush)
        amed, _ = timed(adam, 20, flush)
        out['two_launch_step'] = {'bpr_fwd_bwd_ms': bmed, 'adam_l2_sweep_ms': amed,
                                  'adam_gbs': algorithmic_bytes_adam(t.P.shape[0], D) / (amed * 1e-3) / 1e9}
    except Exception as e:  # noqa: BLE001
        out['two_launch_step'] = {'error': repr(e)}
    _, tensor_peak, _ = peaks()
    try:    # the same dev split on the tcgen05 path (bf16 operands, fp32 accumulate; includes the bf16 packing kernels)
        fn = lambda: _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws, precision=1)
        fn(); torch.cuda.synchronize()
        med, _ = timed(fn, 10, flush)
        tf = 2.0 * R * nI * D / (med * 1e-3) / 1e12
        out['eval_tcgen05'] = {'users_per_s': R / (med * 1e-3), 'rows': R, 'items': nI, 'ms': med, 'tflops': tf,
                               'frac_of_bf16_peak': tf / tensor_peak}
    except Exception as e:  # noqa: BLE001
        out['eval_tcgen05'] = {'error': repr(e)}
    try:    # the same dev split with precision 2: the fp32 path's ranks (bit-identical) from split-bf16 tensor-core scores
        fn = lambda: _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws, precision=2)
        r2 = fn()[0]; torch.cuda.synchronize()
        r0 = _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws, precision=0)[0]
        med, _ = timed(fn, 10, flush)
        out['eval_exact_tc'] = {'users_per_s': R / (med * 1e-3), 'rows': R, 'items': nI, 'ms': med,
                                'tflops_fp32_equivalent': 2.0 * R * nI * D / (med * 1e-3) / 1e12,
                                'ranks_identical_to_fp32_path': bool(torch.equal(r0, r2)),
                                'note': 'includes the operand split kernels, the re-check kernel and the status read-back'}
    except Exception as e:  # noqa: BLE001
        out['eval_exact_tc'] = {'error': repr(e)}
    try:    # BASELINE.json configs[4]-shaped sweep point: many rows x 1M items, where the GEMM dominates
        for d in (64, 128):
            nUs, nIs, Rs = 200_000, 1_000_000, 262_144
            g = torch.Generator(device=dev); g.manual_seed(3407)
            Ub = torch.randn((nUs, d), device=dev, generator=g) / d ** 0.5
            Ib = torch.randn((nIs, d), device=dev, generator=g)
            us = torch.randint(0, nUs, (Rs,), device=dev, generator=g)
            ps = torch.randint(0, nIs, (Rs,), device=dev, generator=g)
            hl = 50
            hp_ = torch.arange(0, (nUs + 1) * hl, hl, device=dev, dtype=torch.int64)
            hi_ = torch.sort(torch.randint(0, nIs, (nUs, hl), device=dev, generator=g), dim=1).values.to(torch.int32).reshape(-1).contiguous()
            ws2 = _lib.Workspace(dev)
            fn = lambda: _lib.eval_rank_topk(Ub, Ib, us, ps, hp_, hi_, ws2, precision=1)
            fn(); torch.cuda.synchronize()
            med, _ = timed(fn, 3)
            tf = 2.0 * Rs * nIs * d / (med * 1e-3) / 1e12
            out['eval_tcgen05_262144x1M_d%d' % d] = {'users_per_s': Rs / (med * 1e-3), 'ms': med, 'tflops': tf,
                                                      'frac_of_bf16_peak': tf / tensor_peak,
                                                      'peak_tflops': tensor_peak}
            fn2 = lambda: _lib.eval_rank_topk(Ub, Ib, us, ps, hp_, hi_, ws2, precision=2)
            r2 = fn2()[0]; torch.cuda.synchronize()
            med2, _ = timed(fn2, 2)
            sub = slice(0, 4096)          # fp32 spot check on a slice (the fp32 path needs ~1.3 s for all rows)
            r0 = _lib.eval_rank_topk(Ub, Ib, us[sub].contiguous(), ps[sub].contiguous(), hp_, hi_, ws2, precision=0)[0]
            out['eval_exact_tc_262144x1M_d%d' % d] = {
                'users_per_s': Rs / (med2 * 1e-3), 'ms': med2, 'tflops_fp32_equivalent': 2.0 * Rs * nIs * d / (med2 * 1e-3) / 1e12,
                'tensor_tflops_issued': 3 * 2.0 * Rs * nIs * d / (med2 * 1e-3) / 1e12,
                'ranks_identical_to_fp32_path_on_4096_rows': bool(torch.equal(r0, r2[sub]))}
            del Ub, Ib, us, ps, hp_, hi_
    except Exception as e:  # noqa: BLE001
        out['eval_tcgen05_sweep'] = {'error': repr(e)}
    try:    # BASELINE.json configs[4]: 1M eval rows x {1M, 2M, 5M, 10M} items, D in {64, 128}, ranks (k = 0) on tcgen05
        sweep = {}
        burst = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))).get('bf16_tflops', 1649.7) \
            if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else 1590.0
        Rs, nUs = 1_000_000, 1_000_000
        for d in (64, 128):
            g = torch.Generator(device=dev); g.manual_seed(3407)
            Ub = torch.randn((nUs, d), device=dev, generator=g) / d ** 0.5
            us = torch.arange(Rs, device=dev, dtype=torch.int64)
            for nIs in (1_000_000, 2_000_000, 5_000_000, 10_000_000):
                Ib = torch.randn((nIs, d), device=dev, generator=g)
                ps = torch.randint(0, nIs, (Rs,), device=dev, generator=g)
                hp_ = torch.arange(0, (nUs + 1) * 50, 50, device=dev, dtype=torch.int64)
                hi_ = torch.sort(torch.randint(0, nIs, (nUs, 50), device=dev, generator=g), dim=1).values.to(torch.int32).reshape(-1).contiguous()
                ws2 = _lib.Workspace(dev)
                fn = lambda: _lib.eval_rank_topk(Ub, Ib, us, ps, hp_, hi_, ws2, precision=1)
                fn(); torch.cuda.synchronize()
                med, _ = timed(fn, 2)
                tf = 2.0 * Rs * nIs * d / (med * 1e-3) / 1e12
                sweep['1Mx%dM_d%d' % (nIs // 1_000_000, d)] = {'users_per_s': Rs / (med * 1e-3), 'ms': med, 'tflops': tf,
                                                               'frac_of_bf16_burst_peak': tf / burst}
                del Ib, ps, hi_
            del Ub
        sweep['note'] = 'embeddings N(0, 1/D), history 50 items per user, seed 3407; timed in isolation -> burst peak %.1f TFLOP/s' % burst
        out['eval_sweep_configs4'] = sweep
    except Exception as e:  # noqa: BLE001
        out['eval_sweep_configs4'] = {'error': repr(e)}
    try:    # LightGCN L=2 on the same graph (BASELINE.json configs[2])
        lg, lrun, ldata = make_model(corpus, dev, 'LightGCN', gcn_layers=2)
        batches = lrun.epoch_batches(ldata['train'])
        def lstep(s=[0]):
            lo = (s[0] % (batches.shape[1] // B)) * B; s[0] += 1
            lg.predict({'user_id': batches[0, lo:lo + B], 'pos_item': batches[1, lo:lo + B], 'neg_items': batches[2, lo:lo + B]})
            lg.optimizer.step()
        for _ in range(5): lstep()
        med, mean = timed(lstep, 30, flush)
        N, nnz = lg.tables.P.shape[0], lg.adj_col.numel()
        Pb = nnz * (4 + 4 + 4 * D) + N * (4 + 4 * D)
        step_bytes = 4 * Pb + 2 * 4 * N * 4 * D + 32 * D * N + 48 * B * D + 12 * B
        spmm = lambda: _lib.csr_spmm(lg.adj_rowptr, lg.adj_col, lg.adj_val, lg.tables.P, Y=lg.layer[0], plan=lg.adj_plan)
        smed, _ = timed(spmm, 20, flush)
        out['lightgcn_L2'] = {'interactions_per_s': B / (med * 1e-3), 'ms_per_step': med, 'nodes': N, 'nnz': nnz,
                              'algorithmic_step_gbs': step_bytes / (med * 1e-3) / 1e9,
                              'spmm_ms': smed, 'spmm_algorithmic_gbs': Pb / (smed * 1e-3) / 1e9,
                              'spmm_frac_of_hbm_peak': Pb / (smed * 1e-3) / 1e9 / hbm_peak,
                              'note': 'no-reuse byte model; the 2.5 MB table is cache-resident, so > 1.0 is possible'}
        del lg, batches
    except Exception as e:  # noqa: BLE001
        out['lightgcn_L2'] = {'error': repr(e)}
    try:    # BASELINE.json configs[3] on ONE GPU: LightGCN L=3 D=128 on the 10M x 2M x 494M-edge power-law graph (65 GB)
        import argparse as _ap
        from scripts.bench_lightgcn_scale import run as lightgcn_scale
        torch.cuda.empty_cache()
        cfg = _ap.Namespace(users=10_000_000, items=2_000_000, edges=500_000_000, dim=128, layers=3, batch=65536, steps=3, warmup=1)
        out['lightgcn_cfg4_10Mx2Mx494M_L3_d128'] = lightgcn_scale(cfg, 0, 1, dev)
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out['lightgcn_cfg4_10Mx2Mx494M_L3_d128'] = {'error': repr(e)}
    try:    # the same two training kernels where HBM really is the bound: 10M users x 2M items, D=128
        nU, nI, d, b = 10_000_000, 2_000_000, 128, 65536
        P = torch.empty((nU + nI, d), device=dev).normal_(0, 0.01)
        M, V, G = torch.zeros_like(P), torch.zeros_like(P), torch.zeros_like(P)
        ws, loss = _lib.Workspace(dev), torch.zeros(1, device=dev)
        u = torch.randint(0, nU, (b,), device=dev); p = torch.randint(0, nI, (b,), device=dev); n = torch.randint(1, nI, (b,), device=dev)
        k = [0]
        touched = _lib.row_map(nU + nI, dev)
        def big():          # the model's train_step on tables this size: wr_bprmf_step_marked
            k[0] += 1
            _lib.bprmf_step(P, M, V, G, u, p, n, nU, k[0], LR, L2, loss, ws, touched=touched)
        def big_dense():    # the same step with the dense sweep (every gradient row read and re-zeroed)
            k[0] += 1
            _lib.bprmf_step(P, M, V, G, u, p, n, nU, k[0], LR, L2, loss, ws)
        adam = lambda: _lib.adam_l2_sweep(P, M, V, G, 1, LR, L2)
        bpr = lambda: _lib.bpr_fwd_bwd(P[:nU], P[nU:], u, p, n, G[:nU], G[nU:], loss, ws)
        big(); torch.cuda.synchronize()
        med, _ = timed(big, 5)
        dmed, _ = timed(big_dense, 5)
        amed, _ = timed(adam, 5)
        bmed, _ = timed(bpr, 5)
        ab = algorithmic_bytes_adam(nU + nI, d)
        out['bprmf_10Mx2M_d128_b65536'] = {
            'interactions_per_s': b / (med * 1e-3), 'ms_per_step': med, 'ms_per_step_dense_sweep': dmed,
            'adam_ms': amed, 'bpr_ms': bmed,
            'step_gbs_row_marked': (ab * 0.75 + algorithmic_bytes_bpr(b, d)) / (med * 1e-3) / 1e9,
            'adam_gbs': ab / (amed * 1e-3) / 1e9, 'adam_frac_of_hbm_peak': ab / (amed * 1e-3) / 1e9 / hbm_peak,
            'bpr_gbs': algorithmic_bytes_bpr(b, d) / (bmed * 1e-3) / 1e9,
            'step_frac_of_hbm_peak': (ab * 0.75 + algorithmic_bytes_bpr(b, d)) / (med * 1e-3) / 1e9 / hbm_peak,
            'dense_step_frac_of_hbm_peak': (ab + algorithmic_bytes_bpr(b, d)) / (dmed * 1e-3) / 1e9 / hbm_peak,
            'note': 'tables 24.6 GB >> L2; dense Adam makes the sweep the whole step.  ms_per_step: row-marked sweep '
                    '(24 B per parameter: the gradient is read only in the rows the batch touched); '
                    'ms_per_step_dense_sweep / adam_ms: the 32 B dense sweep'}
        del P, M, V, G
    except Exception as e:  # noqa: BLE001
        out['bprmf_10Mx2M_d128_b65536'] = {'error': repr(e)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', type=str, default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-budget', type=float, default=12.0, dest='cpu_budget')
    ap.add_argument('--no-extras', action='store_true', dest='no_extras')
    ap.add_argument('--dump-outputs', metavar='DIR', dest='dump_outputs', default=None,
                    help='write the loss and the embedding tables of the last timed step as DIR/<name>.npy (float32)')
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3)
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    import logging
    logging.disable(logging.INFO)
    quiet_stdout()
    if a.impl == 'reference':
        run_reference(a, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device for the sm_100a arm (there is no CPU fallback); '
                         'use --impl reference for the CPU arm')
    if world > 1:
        run_ours_sharded(a, rank, world, local_rank)
    else:
        run_ours(a, rank, world, local_rank)


if __name__ == '__main__':
    main()
