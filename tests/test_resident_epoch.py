"""The resident BPRMF kernels of csrc/epoch_kernel.cu in every form, at every embedding size they are built for.

wr_bprmf_epoch (BaseRunner.fit) and wr_bprmf_ctx_* (train_step_host) run one of three forms, chosen from the table
size, D and the batch capacity: the owner-computes kernel (one grid barrier per step, P double-buffered through G),
the two-barrier kernel, or one wr_bprmf_step launch per batch.  Every test here first asserts, through
wr_bprmf_epoch_form, the form it means to exercise, then compares numbers with one of two references:
  * short epochs (at most 4 steps): a float64 restatement of every step (oracle.bpr_fwd_bwd + oracle.adam_l2_step on
    float64 tensors, Adam's scalars in double as adam_step_scalars computes them);
  * long epochs: the per-step path on the same inputs (bprmf_epoch(..., resident=False)).
Eligibility limits are found by bisecting with the same query, never by restating the shared-memory arithmetic.
"""
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

from oracle import whispr_oracle as O
from tests.helpers import assert_close, ml100k_corpus, model_args
from whisprrec_b200 import _lib
from whisprrec_b200.helpers.BaseRunner import BaseRunner
from whisprrec_b200.models.general.BPRMF import BPRMF
from whisprrec_b200.utils import utils

pytestmark = pytest.mark.gpu
DEV = 'cuda'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIMS = (16, 32, 64, 128, 256)
NU, NI = 700, 900                     # the parity test's 1,600-row table
OWNER, TWO, PER_STEP = _lib.EPOCH_OWNER, _lib.EPOCH_TWO_BARRIER, _lib.EPOCH_PER_STEP
FORM_NAME = {OWNER: 'owner', TWO: 'two_barrier', PER_STEP: 'per_step'}
LR, L2 = 1e-3, 1e-6

# ---- tolerances ----
# Against the per-step path (both sides fp32, the same per-entry arithmetic, gradients summed in another order): the
# suite's parity bar -- losses within 2e-6 relative, P / M / V within 1e-5 relative + 2e-6 of the array's largest value.
STEP_LOSS_RTOL = 2e-6
STEP_RTOL, STEP_ATOL = 1e-5, 2e-6
# Against the float64 chain (4 steps at most): the fp32 kernels round every gather, dot product, gradient sum and Adam
# update.  M, V: |a - b| <= F64_RTOL |b| + F64_ATOL max|b|, the per-step bar.  P gets F64_P_LR more, a share of one
# Adam step lr: where an element's gradient nearly cancels, Adam's direction m / (sqrt(v) + eps) is ill-conditioned and
# fp32 may move that element by a small part of a step more or less than float64 (M and V, linear in the gradient,
# stay tight and catch a wrong gradient: Adam's first steps are ~ lr sign(g) whatever the gradient's scale).
# Measured on a B200 (148 SMs, 1,000 W power limit) over every float64 case of this file, worst of three runs: an
# element used 0.26 of the M bar, 0.14 of the V bar and 0.40 of the P bar, a loss 0.13 of its bar (2.5x margin or more).
# Without F64_P_LR, 1 of ~50,000-100,000 P elements of some cases exceeded the plain bar (by up to 1.8 times it).
F64_RTOL, F64_ATOL, F64_P_LR = 1e-5, 2e-6, 2e-3
F64_LOSS_RTOL = 2e-6

RAN = set()          # (route, form, D) of every call a test checked the numbers of
F64_WORST = {}       # name -> the largest share of the float64 bar a result used


def dv(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope='module')
def ws():
    return _lib.Workspace(DEV)


def grid():
    """CTAs of a resident launch: one per SM (at most WR_EP_MAX_GRID = 256)."""
    return min(torch.cuda.get_device_properties(0).multi_processor_count, 256)


def form(nU, nI, D, B, host_fed=False):
    return _lib.bprmf_epoch_form(nU, nI, D, B, host_fed)


def last_true(pred, lo, hi):
    """The largest x in [lo, hi] with pred(x), for pred true on [lo, x] and false above."""
    assert pred(lo)
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if pred(mid):
            lo = mid
        else:
            hi = mid - 1
    return lo


def owner_batch_limit(nU, nI, D):
    """The largest batch the owner-computes kernel takes on this table (its staged ids share the SM's shared memory
    with the table slice)."""
    return last_true(lambda b: form(nU, nI, D, b) == OWNER, 1, 128 * grid())


def matrix_batch(D, want):
    """A batch that selects `want` on the 1,600-row table: at most 2,048 rows for the owner form, at least 4,096 (and
    past the owner form's limit) for the two-barrier kernel."""
    lim = owner_batch_limit(NU, NI, D)
    return min(2048, lim) if want == OWNER else max(4096, lim + 1)


def table(rows, D, rng, scale=0.1):
    return (rng.randn(rows, D) * scale).astype(np.float32)


def uniform_ids(rng, nU, nI, N):
    return np.stack([rng.randint(0, nU, N), rng.randint(0, nI, N), rng.randint(0, nI, N)]).astype(np.int64)


# ---- the two references ----
def f64_chain(P0, ids, B, nU, t0, lr, l2, state=None):
    """Every step of the epoch in float64: (losses, P, M, V)."""
    P = torch.from_numpy(P0).double()
    M, V = (torch.zeros_like(P), torch.zeros_like(P)) if state is None else \
        (torch.from_numpy(state[0]).double(), torch.from_numpy(state[1]).double())
    losses = []
    for s, lo in enumerate(range(0, ids.shape[1], B)):
        u, i, j = (torch.from_numpy(np.ascontiguousarray(ids[r, lo:lo + B])) for r in range(3))
        loss, gU, gI = O.bpr_fwd_bwd(P[:nU], P[nU:], u, i, j)
        O.adam_l2_step(P, M, V, torch.cat([gU, gI]), t0 + s + 1, lr, l2)      # bias corrections in double
        losses.append(float(loss))
    return np.array(losses), P.numpy(), M.numpy(), V.numpy()


def device_epoch(P0, ids, B, nU, t0, lr, l2, ws, resident=True, state=None):
    """bprmf_epoch on a fresh copy of the state: (losses, P, M, V, G) on the host."""
    P = dv(P0)
    M, V = (torch.zeros_like(P), torch.zeros_like(P)) if state is None else (dv(state[0]), dv(state[1]))
    G = torch.zeros_like(P)
    steps = (ids.shape[1] + B - 1) // B
    losses = torch.full((steps,), -1.0, device=DEV)
    assert _lib.bprmf_epoch(P, M, V, G, dv(ids), B, nU, t0, lr, l2, losses, ws, resident=resident) == steps
    return host(losses), host(P), host(M), host(V), host(G)


def check_f64(got, ref, lr, what):
    (gl, gP, gM, gV), (rl, rP, rM, rV) = got[:4], ref
    assert np.all(gl > 0), f'{what}: a step wrote no loss'
    share = float(np.max(np.abs(gl - rl) / (F64_LOSS_RTOL * np.abs(rl))))
    F64_WORST['loss'] = max(F64_WORST.get('loss', 0.0), share)
    assert share <= 1.0, f'{what}: losses vs float64 {gl} {rl}'
    for name, a, b, extra in (('P', gP, rP, F64_P_LR * lr), ('M', gM, rM, 0.0), ('V', gV, rV, 0.0)):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        err = np.abs(a - b)
        bar = F64_RTOL * np.abs(b) + F64_ATOL * np.max(np.abs(b)) + extra + 1e-30
        share = float(np.max(err / bar))
        F64_WORST[name] = max(F64_WORST.get(name, 0.0), share)
        assert share <= 1.0, (f'{what}: {name} vs float64: {np.count_nonzero(err > bar)} of {err.size} elements out '
                              f'of tolerance; max abs err {err.max():.3e}, max |ref| {np.abs(b).max():.3e}')


def check_vs_per_step(got, ref, what, p_extra=0.0):
    assert np.all(got[0] > 0), f'{what}: a step wrote no loss'
    assert_close(got[0], ref[0], f'{what}: losses vs per-step', rtol=STEP_LOSS_RTOL, atol_scale=0.0)
    for k, name in ((2, 'M'), (3, 'V')):
        assert_close(got[k], ref[k], f'{what}: {name} vs per-step', rtol=STEP_RTOL, atol_scale=STEP_ATOL)
    err = np.abs(got[1].astype(np.float64) - ref[1])
    bar = STEP_RTOL * np.abs(ref[1]) + STEP_ATOL * np.abs(ref[1]).max() + p_extra
    assert np.all(err <= bar), f'{what}: P vs per-step: {np.count_nonzero(err > bar)} elements, max err {err.max():.3e}'


def run_f64_case(P0, ids, B, nU, D, want, ws, what, t0=0, lr=LR, l2=L2):
    """One resident epoch of at most 4 steps against the float64 chain; G comes back zero, no status bit."""
    nI = P0.shape[0] - nU
    assert form(nU, nI, D, B) == want, f'{what}: expected the {FORM_NAME[want]} form'
    assert (ids.shape[1] + B - 1) // B <= 4
    got = device_epoch(P0, ids, B, nU, t0, lr, l2, ws)
    check_f64(got, f64_chain(P0, ids, B, nU, t0, lr, l2), lr, what)
    assert float(np.abs(got[4]).max()) == 0.0, f'{what}: G not handed back zero'
    assert ws.status() == 0
    RAN.add(('device', want, D))
    return got


def run_step_case(P0, ids, B, nU, D, want, ws, what, t0=0, lr=LR, l2=L2, state=None):
    """One epoch in the expected form against the per-step path on the same inputs.  Above the default lr, P gets the
    float64 comparison's allowance of F64_P_LR lr: the per-step bar's absolute term is sized for lr = 1e-3."""
    nI = P0.shape[0] - nU
    assert form(nU, nI, D, B) == want, f'{what}: expected the {FORM_NAME[want]} form'
    got = device_epoch(P0, ids, B, nU, t0, lr, l2, ws, state=state)
    ref = device_epoch(P0, ids, B, nU, t0, lr, l2, ws, resident=False, state=state)
    check_vs_per_step(got, ref, what, F64_P_LR * lr if lr > LR else 0.0)
    assert float(np.abs(got[4]).max()) == 0.0, f'{what}: G not handed back zero'
    assert ws.status() == 0
    RAN.add(('device', want, D))
    return got


# ---- cases aimed at the owner kernel's row map (also run on the two-barrier kernel, in a child process) ----
def case_small_tables(D, want, ws):
    """Fewer rows than CTAs (3 + 5), exactly one row per CTA, one row more: most CTAs own nothing, and one owns
    two rows.  B = 64, the last batch ragged at 1 row."""
    g = grid()
    for nU, nI in ((3, 5), (g // 2, g - g // 2), (g // 2, g - g // 2 + 1)):
        rng = np.random.RandomState(nU + nI + D)
        P0 = table(nU + nI, D, rng)
        ids = uniform_ids(rng, nU, nI, 3 * 64 + 1)
        run_f64_case(P0, ids, 64, nU, D, want, ws, f'{nU}+{nI} rows, D={D}')


def adversarial_ids(rng, nU, nI, N):
    """A mix aimed at local_of (row r -> CTA r % grid, local row r / grid): entries whose user, positive and negative
    rows are congruent mod grid (one CTA owns all three roles), pos == neg, rows k grid - 1 and k grid, the first and
    last row of either table, and a uniform remainder."""
    g = grid()
    ids = uniform_ids(rng, nU, nI, N)
    q = N // 4
    # congruent triples: nU + i = u (mod g), nU + j = u (mod g)
    u = rng.randint(0, nU, q)
    for r in (1, 2):
        base = (u - nU) % g
        k = rng.randint(0, max(1, (nI - base.max()) // g), q)
        it = base + k * g
        it[it >= nI] = base[it >= nI]
        ids[r, :q] = it
    ids[0, :q] = u
    ids[0, q:q + 40] = u[:40]                                   # pos == neg, same congruent user
    ids[2, q:q + 40] = ids[1, q:q + 40]
    ids[2, q + 40:2 * q] = ids[1, q + 40:2 * q]                 # pos == neg, uniform
    # boundary rows of the cyclic map and of the tables
    rows = sorted({r for k in range(1, (nU + nI) // g + 2) for r in (k * g - 1, k * g) if 0 <= r < nU + nI} |
                  {0, nU - 1, nU, nU + nI - 1})
    users = [r for r in rows if r < nU]
    items = [r - nU for r in rows if r >= nU]
    s = slice(2 * q, 3 * q)
    ids[0, s] = rng.choice(users, q)
    ids[1, s] = rng.choice(items, q)
    ids[2, s] = rng.choice(items, q)
    return ids


def case_row_map_ids(D, want, ws):
    rng = np.random.RandomState(100 + D)
    P0 = table(NU + NI, D, rng)
    ids = adversarial_ids(rng, NU, NI, 3 * 1024 + 511)
    run_f64_case(P0, ids, 1024, NU, D, want, ws, f'row-map ids, D={D}')


def case_hot_rows(D, want, ws):
    """One user and one item in every entry: the owning CTAs' lists hold all B entries and every gradient add of the
    step lands on the same shared-memory float4s (the contended 128-bit CAS)."""
    rng = np.random.RandomState(200 + D)
    P0 = table(NU + NI, D, rng)
    N = 3 * 2048 + 1000
    ids = uniform_ids(rng, NU, NI, N)
    ids[0, :] = 5                  # hot user
    ids[1, :] = 17                 # hot positive
    ids[2, ::7] = 17               # and now and then as the negative too
    run_f64_case(P0, ids, 2048, NU, D, want, ws, f'hot rows, D={D}')


# =====================================================================================================================
# device-fed (wr_bprmf_epoch)
# =====================================================================================================================

def test_form_query_is_monotone_and_agrees_with_its_switches():
    """The query itself: the owner form on small batches, the two-barrier kernel above its staging limit, per-step
    launches above 128 x grid rows, for sizes the kernels are not built for and for tables beyond shared memory."""
    g = grid()
    for D in DIMS:
        lim = owner_batch_limit(NU, NI, D)
        assert form(NU, NI, D, lim + 1) == TWO and form(NU, NI, D, 128 * g) == TWO
        assert form(NU, NI, D, 128 * g + 1) == PER_STEP
        assert form(NU, NI, D, 2048, host_fed=True) == TWO          # the host-fed context keeps the two-barrier kernel
        assert form(NU, NI, D, 128 * g + 1, host_fed=True) == PER_STEP
    assert form(NU, NI, 48, 64) == PER_STEP and form(NU, NI, 48, 64, host_fed=True) == PER_STEP
    assert form(4_000_000, 3_000_000, 64, 2048) == PER_STEP


@pytest.mark.parametrize('D', DIMS)
@pytest.mark.parametrize('want', [OWNER, TWO], ids=['owner', 'two_barrier'])
def test_device_fed_form_matrix(want, D, ws):
    """Both resident forms at every D on the 1,600-row table: 4 steps (the last ragged) against float64, then a second
    epoch from the written-back state (adam_t0 = steps) against the per-step path."""
    B = matrix_batch(D, want)
    rng = np.random.RandomState(10 * D + want)
    P0 = table(NU + NI, D, rng)
    ids = uniform_ids(rng, NU, NI, 3 * B + B // 3)
    first = run_f64_case(P0, ids, B, NU, D, want, ws, f'{FORM_NAME[want]} D={D} B={B}')
    ids2 = uniform_ids(rng, NU, NI, 5 * B + 17)
    run_step_case(first[1], ids2, B, NU, D, want, ws, f'{FORM_NAME[want]} D={D} 2nd epoch', t0=4,
                  state=(first[2], first[3]))


@pytest.mark.parametrize('D', [16, 64, 256])
def test_owner_tables_smaller_than_and_around_the_grid(D, ws):
    case_small_tables(D, OWNER, ws)


@pytest.mark.parametrize('D', DIMS)
def test_owner_row_map_congruent_and_boundary_ids(D, ws):
    case_row_map_ids(D, OWNER, ws)


@pytest.mark.parametrize('D', [16, 64, 256])
def test_owner_hot_user_and_item_in_every_entry(D, ws):
    case_hot_rows(D, OWNER, ws)


def test_owner_zipf_items_ml1m_shape(ws):
    """The bench's shape (6,040 users x 3,706 items, D = 64, B = 2,048) with Zipf-distributed items, 23 steps."""
    rng = np.random.RandomState(61)
    nU, nI, D, B = 6040, 3706, 64, 2048
    P0 = table(nU + nI, D, rng)
    w = 1.0 / np.arange(1, nI + 1) ** 1.1
    w /= w.sum()
    N = 22 * B + 300
    ids = np.stack([rng.randint(0, nU, N), rng.choice(nI, N, p=w), rng.choice(nI, N, p=w)]).astype(np.int64)
    want = form(nU, nI, D, B)
    assert want != PER_STEP
    run_step_case(P0, ids, B, nU, D, want, ws, f'zipf ml-1m shape ({FORM_NAME[want]})')


@pytest.mark.parametrize('D,B,N', [(64, 1, 5), (16, 31, 31 * 6 + 1), (256, 31, 31 * 4 + 1), (32, 33, 33 * 12 + 1),
                                   (128, 100, 100 * 10 + 1), (64, 1000, 1000 * 8 + 1), (64, 2048, 2048 * 14 + 1)])
def test_owner_small_and_ragged_batches_odd_step_counts(D, B, N, ws):
    """B = 1, 31, 33, 100, ...; step counts 5, 7, 5, 13, 11, 9, 15 (odd, and no multiple of a staging depth 2-4 or of
    WR_EP_PART_DEPTH = 4); every last batch is 1 row."""
    rng = np.random.RandomState(D + B)
    P0 = table(NU + NI, D, rng)
    run_step_case(P0, uniform_ids(rng, NU, NI, N), B, NU, D, OWNER, ws, f'D={D} B={B} N={N}')


def test_owner_f64_single_entry_batches(ws):
    """B = 1: four steps of one entry each (one CTA owns the user, others the items), against float64."""
    rng = np.random.RandomState(3)
    P0 = table(NU + NI, 64, rng)
    run_f64_case(P0, uniform_ids(rng, NU, NI, 4), 1, NU, 64, OWNER, ws, 'B=1')


def test_owner_long_epoch_every_ring_wraps(ws):
    """501 steps of 32 rows (the last one 7): the staging, loss-partial and duty rings wrap many times.  (The
    two-barrier kernel runs the same epoch in test_two_barrier_kernel_at_the_owner_shapes.)"""
    rng = np.random.RandomState(500)
    P0 = table(NU + NI, 32, rng)
    run_step_case(P0, uniform_ids(rng, NU, NI, 32 * 500 + 7), 32, NU, 32, OWNER, ws, '501 steps (owner)')


def test_owner_at_staging_depths_4_3_and_2(ws):
    """The owner kernel stages up to 4 steps of ids; with larger batches fewer fit beside the table slice.  With L the
    owner form's batch limit (depth 2: the slice plus 3 x 24 bytes per id slot fill the SM), a depth-d launch needs
    the slice plus (d + 1) x 24 bytes per id slot, so batches <= 0.55 L stage 4 steps, batches in (0.6 (L + 32),
    0.75 L] stage 3, and L stages 2.  Seven steps each."""
    D = 64
    lim = owner_batch_limit(NU, NI, D)
    assert lim >= 1024          # (large enough for the three ranges to be distinct after rounding to 32)
    for B in (int(0.55 * lim) // 32 * 32, int(0.74 * lim) // 32 * 32, lim):
        rng = np.random.RandomState(B)
        P0 = table(NU + NI, D, rng)
        run_step_case(P0, uniform_ids(rng, NU, NI, 6 * B + 1), B, NU, D, OWNER, ws, f'owner B={B} (limit {lim})')


def test_eligibility_limits_both_sides_equal_the_per_step_path(ws):
    """The last table size and batch each resident form accepts, and one more: each side gives the per-step numbers."""
    g = grid()
    cases = []
    # owner form, table rows (B = 2,048, D = 256): one row more is the two-barrier kernel
    n = last_true(lambda nI: form(NU, nI, 256, 2048) == OWNER, 1, 1 << 20)
    cases += [(NU, n, 256, 2048, OWNER), (NU, n + 1, 256, 2048, TWO)]
    # two-barrier kernel, table rows (B = 4,096, D = 64): one row more is per-step launches
    n = last_true(lambda nI: form(NU, nI, 64, 4096) == TWO, 1, 1 << 24)
    cases += [(NU, n, 64, 4096, TWO), (NU, n + 1, 64, 4096, PER_STEP)]
    # owner form, batch (1,600 rows, D = 64)
    lim = owner_batch_limit(NU, NI, 64)
    cases += [(NU, NI, 64, lim, OWNER), (NU, NI, 64, lim + 1, TWO)]
    # two-barrier kernel, batch (1,600 rows, D = 32): 128 rows per CTA
    cases += [(NU, NI, 32, 128 * g, TWO), (NU, NI, 32, 128 * g + 1, PER_STEP)]
    for nU, nI, D, B, want in cases:
        rng = np.random.RandomState(nI + B)
        P0 = table(nU + nI, D, rng, 0.05)
        run_step_case(P0, uniform_ids(rng, nU, nI, 4 * B + 1), B, nU, D, want, ws,
                      f'{nU}+{nI} rows D={D} B={B} ({FORM_NAME[want]})')


@pytest.mark.parametrize('want', [OWNER, TWO], ids=['owner', 'two_barrier'])
@pytest.mark.parametrize('l2,t0,lr', [(0.0, 0, 1e-3), (1e-2, 0, 1e-3), (1e-6, 10 ** 6, 1e-3), (1e-6, 5, 3e-2)],
                         ids=['l2=0', 'l2=1e-2', 't0=1e6', 'lr=3e-2'])
def test_adam_scalars(want, l2, t0, lr, ws):
    """l2 = 0 and 1e-2, Adam's t continuing from 10^6 (both bias corrections ~ 1): 4 steps vs float64.  lr = 3e-2: 7
    steps vs the per-step path (at 30 times the default step, fp32's rounding of P feeds back into later gradients:
    measured, M and V of a few elements left the float64 bar by up to 1.4 times it)."""
    D = 64
    B = matrix_batch(D, want)
    rng = np.random.RandomState(int(l2 * 1e6) + t0 % 1000 + want)
    P0 = table(NU + NI, D, rng)
    what = f'{FORM_NAME[want]} l2={l2} t0={t0} lr={lr}'
    if lr == LR:
        run_f64_case(P0, uniform_ids(rng, NU, NI, 3 * B + 5), B, NU, D, want, ws, what, t0=t0, lr=lr, l2=l2)
    else:
        run_step_case(P0, uniform_ids(rng, NU, NI, 6 * B + 5), B, NU, D, want, ws, what, t0=t0, lr=lr, l2=l2)


def _child(env, code, marker):
    r = subprocess.run([sys.executable, '-c', code], cwd=ROOT, env=dict(os.environ, **env), capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and marker in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_two_barrier_kernel_at_the_owner_shapes():
    """WR_EPOCH_KERNEL=two_barrier (read once per process, hence the child): the small tables, row-map ids and hot rows
    above on the two-barrier kernel, which the owner form would otherwise take."""
    code = ('import torch; from whisprrec_b200 import _lib; from tests import test_resident_epoch as t\n'
            'ws = _lib.Workspace(torch.device("cuda:0"))\n'
            'for D in t.DIMS:\n'
            '    t.case_small_tables(D, t.TWO, ws); t.case_row_map_ids(D, t.TWO, ws); t.case_hot_rows(D, t.TWO, ws)\n'
            'rng = t.np.random.RandomState(5)\n'
            't.run_step_case(t.table(t.NU + t.NI, 32, rng), t.uniform_ids(rng, t.NU, t.NI, 32 * 500 + 7), 32, t.NU, 32,'
            ' t.TWO, ws, "501 steps (two_barrier)")\n'
            'print("two-barrier shapes ok")\n')
    _child({'WR_EPOCH_KERNEL': 'two_barrier'}, code, 'two-barrier shapes ok')
    for D in DIMS:
        RAN.add(('device', TWO, D))


# =====================================================================================================================
# host-fed (wr_bprmf_ctx_*)
# =====================================================================================================================

def host_fed_vs_device_steps(D, want, ws, nU=NU, nI=NI, steps=24):
    """A BprmfContext stream (pinned and pageable ids, wait = 0 / 1 / 2, losses collected 8 steps later) against the
    same batches through wr_bprmf_step; P / M / V after the stream is closed."""
    Bmax = 2048
    assert form(nU, nI, D, Bmax, host_fed=True) == want, f'host-fed D={D}: expected {FORM_NAME[want]}'
    rng = np.random.RandomState(D + 7 * want)
    P0 = table(nU + nI, D, rng)
    Pa, Pb = dv(P0), dv(P0)
    Ma, Va, Ga, Mb, Vb, Gb = (torch.zeros_like(Pa) for _ in range(6))
    sizes = [Bmax if k % 5 else 1 + 97 * k for k in range(steps)]
    batches = [uniform_ids(rng, nU, nI, B) for B in sizes]
    ref = []
    lb = torch.zeros(1, device=DEV)
    for k, ids in enumerate(batches):
        d = dv(ids)
        _lib.bprmf_step(Pb, Mb, Vb, Gb, d[0], d[1], d[2], nU, k + 1, LR, L2, lb, ws)
        ref.append(float(lb[0]))
    ctx = _lib.BprmfContext(Pa, Ma, Va, Ga, nU, LR, L2, ws)
    keep = []
    for k, ids in enumerate(batches):
        buf = torch.from_numpy(ids).pin_memory() if k % 3 == 0 else torch.from_numpy(ids)
        keep.append(buf)                        # pinned ids are read in place until their step is complete
        wait = (0, 0, 1, 0, 2)[k % 5]
        loss = ctx.step(buf.data_ptr(), ids.shape[1], k + 1, wait)
        if wait:
            assert loss == pytest.approx(ref[k], rel=STEP_LOSS_RTOL), (D, k)
        if k >= 8:
            assert ctx.wait(k - 8) == pytest.approx(ref[k - 8], rel=STEP_LOSS_RTOL), (D, k - 8)
    for k in range(steps - 8, steps):
        assert ctx.wait(k, 2) == pytest.approx(ref[k], rel=STEP_LOSS_RTOL), (D, k)
    ctx.sync()
    for name, a, b in (('P', Pa, Pb), ('M', Ma, Mb), ('V', Va, Vb)):
        assert_close(host(a), host(b), f'host-fed D={D} {name}', rtol=STEP_RTOL, atol_scale=STEP_ATOL)
    assert float(Ga.abs().max()) == 0.0
    ctx.close()
    assert ws.status() == 0


@pytest.mark.parametrize('D', DIMS)
def test_host_fed_two_barrier_every_dim(D, ws):
    host_fed_vs_device_steps(D, TWO, ws)
    RAN.add(('host', TWO, D))


def test_host_fed_owner_every_dim():
    """WR_CTX_KERNEL=owner puts the host-fed context on the owner-computes kernel (read once per process)."""
    code = ('import torch; from whisprrec_b200 import _lib; from tests import test_resident_epoch as t\n'
            'ws = _lib.Workspace(torch.device("cuda:0"))\n'
            'for D in t.DIMS: t.host_fed_vs_device_steps(D, t.OWNER, ws)\n'
            'print("host-fed owner ok")\n')
    _child({'WR_CTX_KERNEL': 'owner'}, code, 'host-fed owner ok')
    for D in DIMS:
        RAN.add(('host', OWNER, D))


def test_host_fed_stream_across_routes_numbers_every_step(ws):
    """model.train_step_host through a growing batch: 2,048 -> 3,000 -> 5,000 rows (relaunches at a larger capacity
    with wait = 0 steps in flight), then a batch above 128 x grid (per-step launches), then 2,048 again, an idle exit
    and relaunch.  Pinned and pageable ids; every loss collected later by host_step_loss(k) equals
    model.train_step's on the same batch, and so do P / M / V at the end."""
    corpus = ml100k_corpus()
    nU, nI = corpus.n_users, corpus.n_items
    big = 128 * grid() + 1
    assert form(nU, nI, 64, 2048, host_fed=True) == TWO and form(nU, nI, 64, 5000, host_fed=True) == TWO
    assert form(nU, nI, 64, big, host_fed=True) == PER_STEP
    models = []
    for _ in range(2):
        args = model_args(BPRMF, lr=LR, l2=L2)
        utils.init_seed(3407)
        m = BPRMF(args, corpus).to(DEV)
        m.fuse()
        m.optimizer = BaseRunner(args)._build_optimizer(m)
        models.append(m)
    sizes = [2048] * 3 + [3000] * 2 + [5000] * 2 + [big, 2048, 2048, big, big] + [2048] * 6 + ['idle'] + [2048] * 3
    rng = np.random.RandomState(21)
    batches = [None if B == 'idle' else np.stack([rng.randint(0, nU, B), rng.randint(1, nI, B), rng.randint(1, nI, B)])
               .astype(np.int64) for B in sizes]
    ref = []
    for ids in batches:
        if ids is not None:
            d = dv(ids)
            ref.append(float(models[1].train_step({'user_id': d[0], 'pos_item': d[1], 'neg_items': d[2]})))
    keep, k = [], 0
    for n, ids in enumerate(batches):
        if ids is None:
            time.sleep(0.05)                   # > the kernel's 5 ms idle limit: it writes its state back and leaves
            continue
        pinned = n % 2 or ids.shape[1] == big          # (pageable ids on the per-step route: the next test)
        buf = torch.from_numpy(ids).pin_memory() if pinned else torch.from_numpy(ids)
        keep.append(buf)
        wait = 1 if n in (9, 17) else 0
        loss = models[0].train_step_host(buf, wait=wait)
        if wait:
            assert loss == pytest.approx(ref[k], rel=STEP_LOSS_RTOL), k
        if k >= 5:
            assert models[0].host_step_loss(k - 5) == pytest.approx(ref[k - 5], rel=STEP_LOSS_RTOL), k - 5
        k += 1
    for j in range(k - 5, k):
        assert models[0].host_step_loss(j) == pytest.approx(ref[j], rel=STEP_LOSS_RTOL), j
    models[0].quiesce()
    for name in ('P', 'M', 'V'):
        assert_close(host(getattr(models[0].tables, name)), host(getattr(models[1].tables, name)), name,
                     rtol=STEP_RTOL, atol_scale=STEP_ATOL)
    assert float(models[0].tables.G.abs().max()) == 0.0
    assert models[0].tables.ws.status() == 0
    RAN.update({('host', TWO, 64), ('host', PER_STEP, 64)})


def test_host_fed_table_that_never_goes_resident(ws):
    """D = 48 has no resident kernel: every step is a per-step launch.  wait = 0 steps, their losses collected later through wr_bprmf_ctx_wait, equal wr_bprmf_step on the same batches."""
    nU, nI, D, B = 300, 500, 48, 700
    assert form(nU, nI, D, B, host_fed=True) == PER_STEP
    rng = np.random.RandomState(48)
    P0 = table(nU + nI, D, rng)
    Pa, Pb = dv(P0), dv(P0)
    Ma, Va, Ga, Mb, Vb, Gb = (torch.zeros_like(Pa) for _ in range(6))
    batches = [uniform_ids(rng, nU, nI, B - 13 * (k % 3)) for k in range(20)]
    ref, lb = [], torch.zeros(1, device=DEV)
    for k, ids in enumerate(batches):
        d = dv(ids)
        _lib.bprmf_step(Pb, Mb, Vb, Gb, d[0], d[1], d[2], nU, k + 1, LR, L2, lb, ws)
        ref.append(float(lb[0]))
    ctx = _lib.BprmfContext(Pa, Ma, Va, Ga, nU, LR, L2, ws)
    keep = []
    for k, ids in enumerate(batches):
        buf = torch.from_numpy(ids).pin_memory()
        keep.append(buf)
        ctx.step(buf.data_ptr(), ids.shape[1], k + 1, wait=0)
        if k >= 6:
            assert ctx.wait(k - 6) == pytest.approx(ref[k - 6], rel=STEP_LOSS_RTOL), k - 6
    for k in range(14, 20):
        assert ctx.wait(k, 2) == pytest.approx(ref[k], rel=STEP_LOSS_RTOL), k
    ctx.sync()
    torch.cuda.synchronize()
    for name, a, b in (('P', Pa, Pb), ('M', Ma, Mb), ('V', Va, Vb)):
        assert_close(host(a), host(b), f'{name}', rtol=STEP_RTOL, atol_scale=STEP_ATOL)
    ctx.close()
    assert ws.status() == 0
    RAN.add(('host', PER_STEP, D))


def test_host_fed_pageable_ids_on_the_per_step_route(ws):
    """model.train_step_host with pageable ids on a batch above 128 x grid rows (per-step launches): the ids are
    collated into the context's pinned ring as on the resident route; then resident steps continue the stream."""
    corpus = ml100k_corpus()
    nU, nI = corpus.n_users, corpus.n_items
    big = 128 * grid() + 1
    assert form(nU, nI, 64, big, host_fed=True) == PER_STEP
    models = []
    for _ in range(2):
        args = model_args(BPRMF, lr=LR, l2=L2)
        utils.init_seed(3407)
        m = BPRMF(args, corpus).to(DEV)
        m.fuse()
        m.optimizer = BaseRunner(args)._build_optimizer(m)
        models.append(m)
    rng = np.random.RandomState(22)
    for k, B in enumerate([big, big, 2048, big, 2048]):
        ids = np.stack([rng.randint(0, nU, B), rng.randint(1, nI, B), rng.randint(1, nI, B)]).astype(np.int64)
        loss = models[0].train_step_host(torch.from_numpy(ids), wait=1 + k % 2)          # pageable
        d = dv(ids)
        ref = float(models[1].train_step({'user_id': d[0], 'pos_item': d[1], 'neg_items': d[2]}))
        assert loss == pytest.approx(ref, rel=STEP_LOSS_RTOL), k
        assert models[0].host_step_loss(k) == pytest.approx(ref, rel=STEP_LOSS_RTOL), k
    models[0].quiesce()
    for name in ('P', 'M', 'V'):
        assert_close(host(getattr(models[0].tables, name)), host(getattr(models[1].tables, name)), name,
                     rtol=STEP_RTOL, atol_scale=STEP_ATOL)
    assert models[0].tables.ws.status() == 0


# =====================================================================================================================

def test_every_form_ran(request):
    """Each form at each D on each route was exercised above, and the per-step route on both (when the whole module
    ran); prints the largest share of the float64 bar any result used."""
    print('float64 bar used at most:', {k: float(f'{v:.3g}') for k, v in sorted(F64_WORST.items())})
    if request.config.getoption('keyword') or any('::' in a for a in request.config.args):
        pytest.skip('only part of the module was selected')
    expected = {(route, f, D) for route in ('device', 'host') for f in (OWNER, TWO) for D in DIMS}
    missing = expected - RAN
    assert not missing, sorted(missing)
    assert {r for r, f, _ in RAN if f == PER_STEP} == {'device', 'host'}
