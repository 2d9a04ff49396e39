"""The single-launch step's grid barrier (per-CTA arrival lines keyed by a launch generation, no reset between launches)
over many consecutive launches of different grid sizes on ONE workspace, interleaved with the resident epoch kernel, and
the traced instantiation (wr_debug_step_trace) against the untraced one.  Needs a B200."""
import numpy as np
import pytest
import torch

from tests.helpers import assert_close
from whisprrec_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = 'cuda'
# (50 + 70) x 16 runs a handful of CTAs, (500 + 700) x 64 more CTAs (100) than threads per CTA (96), the bench shape one
# CTA per SM, (40,000 + 60,000) x 64 several Adam passes per thread
SHAPES = [(50, 70, 16, 33), (500, 700, 64, 2048), (6040, 3706, 64, 2048), (40000, 60000, 64, 8192)]


def within(a, b, rtol=1e-5, atol_scale=2e-6):
    """|a-b| <= rtol |b| + atol_scale max|b| on the device (the tolerance of the two-kernel comparison in test_gpu_parity)."""
    return bool(((a - b).abs() <= rtol * b.abs() + atol_scale * float(b.abs().max())).all())


class Tables:
    def __init__(self, nU, nI, D, B, seed):
        g = torch.Generator(device=DEV)
        g.manual_seed(seed)
        self.nU, self.nI, self.B = nU, nI, B
        self.P = torch.randn((nU + nI, D), device=DEV, generator=g) * 0.1
        self.M, self.V, self.G = (torch.zeros_like(self.P) for _ in range(3))
        self.ref = [torch.zeros_like(self.P) for _ in range(4)]
        self.loss, self.ref_loss = torch.zeros(1, device=DEV), torch.zeros(1, device=DEV)
        self.g = g

    def batch(self):
        g = self.g
        return (torch.randint(0, self.nU, (self.B,), device=DEV, generator=g),
                torch.randint(0, self.nI, (self.B,), device=DEV, generator=g),
                torch.randint(1, self.nI, (self.B,), device=DEV, generator=g))


def test_consecutive_steps_of_different_grids_share_one_workspace():
    ws = _lib.Workspace(DEV)
    tabs = [Tables(*s, seed=k) for k, s in enumerate(SHAPES)]
    # a resident epoch on the same workspace every few steps: its barrier words must not disturb the step's, nor the reverse
    rng = np.random.RandomState(3)
    eU, eI, eD, eN, eB = 500, 700, 64, 5000, 2048
    eP0 = torch.from_numpy((rng.randn(eU + eI, eD) * 0.1).astype(np.float32)).to(DEV)
    ids = torch.from_numpy(np.stack([rng.randint(0, eU, eN), rng.randint(0, eI, eN),
                                     rng.randint(1, eI, eN)]).astype(np.int64)).to(DEV)
    e_steps = (eN + eB - 1) // eB
    rP = eP0.clone()
    rM, rV, rG = (torch.zeros_like(rP) for _ in range(3))
    r_losses = torch.zeros(e_steps, device=DEV)
    for s in range(e_steps):
        lo, hi = s * eB, min(eN, (s + 1) * eB)
        _lib.bpr_fwd_bwd(rP[:eU], rP[eU:], ids[0, lo:hi].contiguous(), ids[1, lo:hi].contiguous(),
                         ids[2, lo:hi].contiguous(), rG[:eU], rG[eU:], r_losses[s:s + 1], ws)
        _lib.adam_l2_sweep(rP, rM, rV, rG, s + 1, 1e-3, 1e-6)
    calls = 0
    for rnd in range(80):
        for t in tabs:
            step = rnd + 1
            user, pos, neg = t.batch()
            Pb, Mb, Vb, Gb = t.ref
            Pb.copy_(t.P); Mb.copy_(t.M); Vb.copy_(t.V)
            _lib.bprmf_step(t.P, t.M, t.V, t.G, user, pos, neg, t.nU, step, 1e-3, 1e-6, t.loss, ws)
            _lib.bpr_fwd_bwd(Pb[:t.nU], Pb[t.nU:], user, pos, neg, Gb[:t.nU], Gb[t.nU:], t.ref_loss, ws)
            _lib.adam_l2_sweep(Pb, Mb, Vb, Gb, step, 1e-3, 1e-6)
            calls += 1
            what = f'call {calls} ({t.nU}+{t.nI})x{t.P.shape[1]}'
            assert float(t.loss) == pytest.approx(float(t.ref_loss), rel=2e-6), what
            assert float(t.G.abs().max()) == 0.0, what
            assert within(t.P, Pb), what + ' P'
            assert within(t.M, Mb, atol_scale=1e-6) and within(t.V, Vb, atol_scale=1e-6), what + ' M / V'
        if rnd % 10 == 9:
            eP = eP0.clone()
            eM, eV, eG = (torch.zeros_like(eP) for _ in range(3))
            e_losses = torch.zeros(e_steps, device=DEV)
            assert _lib.bprmf_epoch(eP, eM, eV, eG, ids, eB, eU, 0, 1e-3, 1e-6, e_losses, ws) == e_steps
            assert_close(e_losses.cpu().numpy(), r_losses.cpu().numpy(), f'epoch losses after {calls} steps', rtol=2e-6)
            assert within(eP, rP), f'epoch P after {calls} steps'
    assert calls >= 300
    assert ws.status() == 0


def test_traced_step_equals_untraced_step():
    nU, nI, D, B = 6040, 3706, 64, 2048
    ws = _lib.Workspace(DEV)
    t = Tables(nU, nI, D, B, seed=11)
    lib = _lib.load()
    trace = torch.zeros((2048, 8), dtype=torch.int64, device=DEV)
    for step in range(1, 4):
        user, pos, neg = t.batch()
        P0, M0, V0 = t.P.clone(), t.M.clone(), t.V.clone()
        _lib.bprmf_step(t.P, t.M, t.V, t.G, user, pos, neg, nU, step, 1e-3, 1e-6, t.loss, ws)
        Pb, Mb, Vb, Gb = t.ref
        Pb.copy_(P0); Mb.copy_(M0); Vb.copy_(V0)
        trace.zero_()
        _lib.check(lib.wr_debug_step_trace(trace.data_ptr()))
        try:
            _lib.bprmf_step(Pb, Mb, Vb, Gb, user, pos, neg, nU, step, 1e-3, 1e-6, t.ref_loss, ws)
        finally:
            _lib.check(lib.wr_debug_step_trace(None))
        assert float(t.loss) == float(t.ref_loss)            # CTA partials summed in CTA order, same grid
        assert within(Pb, t.P) and within(Mb, t.M, atol_scale=1e-6) and within(Vb, t.V, atol_scale=1e-6)
        assert float(Gb.abs().max()) == 0.0
        st = trace.cpu().numpy().astype(np.int64)
        st = st[st[:, 0] != 0]
        assert 1 <= len(st) <= torch.cuda.get_device_properties(0).multi_processor_count
        assert (st > 0).all() and (np.diff(st, axis=1) >= 0).all()
    assert ws.status() == 0
