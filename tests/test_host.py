"""Host-side logic and the C-ABI surface, CPU only (no kernel is launched here)."""
import argparse
import ctypes
import hashlib
import os
import re

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import whispr_oracle as O
from tests.helpers import load, ml100k_corpus, model_args
from whisprrec_b200 import _lib
from whisprrec_b200 import main as wr_main
from whisprrec_b200.helpers.BaseReader import BaseReader
from whisprrec_b200.helpers.BaseRunner import BaseRunner, dataloader_draws
from whisprrec_b200.models.general.BPRMF import BPRMF
from whisprrec_b200.models.general.LightGCN import LightGCN, build_norm_adj_csr
from whisprrec_b200.utils import utils

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the unmodified reference (HeyWeCome/WhisprRec, with data/ml-100k): the interchange tests run its code
REFERENCE = os.environ.get('WHISPRREC_REFERENCE', '')
REF_SRC, REF_DATA = os.path.join(REFERENCE, 'src'), os.path.join(REFERENCE, 'data') + os.sep
needs_reference = pytest.mark.skipif(not REFERENCE or not os.path.exists(os.path.join(REF_SRC, 'models', 'general', 'BPRMF.py')),
                                     reason='needs a checkout of the unmodified reference (set WHISPRREC_REFERENCE)')


def test_library_exports_every_declared_symbol():
    """The header is the contract: every wr_* it declares must be exported, and bound with a signature."""
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    header = open(os.path.join(ROOT, 'include', 'whisprrec_b200.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(wr_[a-z0-9_]+)\s*\(', header))
    assert len(declared) >= 14
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib.wr_version.restype = ctypes.c_int
    assert lib.wr_version() == 100
    lib.wr_workspace_bytes.restype = ctypes.c_size_t
    assert 1024 < lib.wr_workspace_bytes() < (1 << 20)
    lib.wr_error_string.restype = ctypes.c_char_p
    assert b'NULL' in lib.wr_error_string(-1)


def test_argument_errors_need_no_gpu():
    """NULL / size / dimension checks run before any CUDA call."""
    lib = _lib.load()
    assert lib.wr_adam_l2_sweep(None, None, None, None, 10, 0.0, 0.9, 0.999, 1e-8, 1e-3, 1.0, None, None) == -1
    assert lib.wr_bpr_fwd_bwd(16, 16, 16, 16, 16, 8, 6, 4, 4, 1e-10, 1.0, 16, 16, 16, 0, 16, None) == -3   # D=6
    assert lib.wr_bpr_fwd_bwd(16, 16, 16, 16, 16, 0, 8, 4, 4, 1e-10, 1.0, 16, 16, 16, 0, 16, None) == -2   # B=0
    assert lib.wr_bpr_fwd_bwd(16, 20, 16, 16, 16, 8, 8, 4, 4, 1e-10, 1.0, 16, 16, 16, 0, 16, None) == -5   # align
    assert lib.wr_eval_rank_topk(16, 16, 16, 16, 4, 4, 4, 64, 16, 16, 33, 0, 16, 16, 16, 16, None, None, 16, None) == -4
    assert lib.wr_eval_rank_topk(16, 16, 16, 16, 4, 4, 4, 64, 16, 16, 0, 7, None, None, 16, 16, None, None, 16, None) == -6
    assert lib.wr_eval_rank_topk(16, 16, 16, 16, 4, 4, 4, 32, 16, 16, 0, 1, None, None, 16, 16, None, 1024, 16, None) == -3   # tensor-core path: D in {64,128}
    assert lib.wr_eval_scratch_bytes(1000, 5000, 64, 0) == 0 and lib.wr_eval_scratch_bytes(1000, 5000, 64, 1) >= (1000 + 5000) * 128
    # the entry points added for the sampler, the epoch loop and the multi-GPU path check their arguments first too
    assert lib.wr_neg_sample_scratch_bytes(0, 100) == 0 and lib.wr_neg_sample_scratch_bytes(1000, 2) == 0
    small, big = lib.wr_neg_sample_scratch_bytes(10_000, 3706), lib.wr_neg_sample_scratch_bytes(1_000_000, 3706)
    assert 0 < small < big and big > 1_000_000 * 12
    assert lib.wr_neg_sample_mt19937(None, 0, 10, 16, 4, 100, 16, 16, 16, None, None, 16, 1 << 20, 16, None) == -1
    assert lib.wr_bprmf_epoch(16, 16, 16, 16, None, 100, 10, 8, 4, 4, 1e-10, 1e-3, 0.0, 0.9, 0.999, 1e-8, 0, 16, None, 0, 16, None) == -1
    assert lib.wr_bprmf_epoch(16, 16, 16, 16, 16, 100, 0, 8, 4, 4, 1e-10, 1e-3, 0.0, 0.9, 0.999, 1e-8, 0, 16, None, 0, 16, None) == -2
    assert lib.wr_bprmf_epoch_scratch_bytes(100, 10) == 10 * 32 and lib.wr_bprmf_epoch_scratch_bytes(0, 10) == 0
    assert lib.wr_bprmf_epoch_form(0, 900, 64, 2048, 0) == -2 and lib.wr_bprmf_epoch_form(700, 0, 64, 2048, 1) == -2
    assert lib.wr_bprmf_epoch_form(700, 900, 64, 0, 0) == -2 and lib.wr_bprmf_epoch_form(700, 900, 64, -5, 1) == -2
    assert lib.wr_bprmf_epoch_form(700, 900, 6, 2048, 0) == -3 and lib.wr_bprmf_epoch_form(700, 900, 0, 2048, 1) == -3
    assert lib.wr_csr_build(None, 16, 5, 3, 3, 16, 16, 16, 16, 1 << 30, 16, None) == -1
    assert lib.wr_csr_build(16, 16, 0, 3, 3, 16, 16, 16, 16, 1 << 30, 16, None) == -2
    assert lib.wr_csr_build(16, 16, 5, 3, 3, 16, 16, 16, 16, 8, 16, None) == -2          # scratch too small
    assert lib.wr_csr_build_scratch_bytes(5) >= 2 * 5 * 8 and lib.wr_csr_build_scratch_bytes(0) == 0
    assert lib.wr_bprmf_ctx_wait(None, 0, 1, None) == -1 and lib.wr_bprmf_ctx_sync(None) == -1
    assert lib.wr_allgather_shards(None, 16, 64, None) == -1
    assert lib.wr_inbox_scatter(None, 16, 16, 2, 100, 64, None) == -1
    assert lib.wr_inbox_scatter(16, 16, 16, 9, 100, 64, None) == -2          # more ranks than one box holds
    assert lib.wr_topk_merge(16, 16, 2, 10, 33, 16, 16, None) == -4
    assert lib.wr_peer_barrier(None, 2, 0, 1, None, None, 0, None, None, None) == -1
    assert lib.wr_bprmf_step_sharded_supported(4873, 64) == 1 and lib.wr_bprmf_step_sharded_supported(6_000_000, 128) == 0
    # the sparse-gradient entry points (row map) and the copy-engine pushes
    assert lib.wr_mark_rows(16, 16, 16, 8, 10, 7, None, None) == -1
    assert lib.wr_mark_rows(16, 16, 16, 0, 10, 7, 16, None) == -2
    assert lib.wr_adam_l2_sweep_marked(16, 16, 16, 16, 100, 64, None, 0.0, 0.9, 0.999, 1e-8, 1e-3, 1.0, None, None) == -1
    assert lib.wr_adam_l2_sweep_marked(16, 16, 16, 16, 100, 6, 16, 0.0, 0.9, 0.999, 1e-8, 1e-3, 1.0, None, None) == -3
    assert lib.wr_adam_l2_sweep_marked(16, 16, 16, 20, 100, 64, 16, 0.0, 0.9, 0.999, 1e-8, 1e-3, 1.0, None, None) == -5
    assert lib.wr_inbox_scatter_marked(None, 16, 16, 2, 100, 64, 16, None) == -1
    assert lib.wr_bprmf_step_marked(16, 16, 16, 16, None, 16, 16, 16, 8, 64, 10, 7, 1e-10, 0.0, 0.9, 0.999, 1e-8, 1e-3, 1.0,
                                    None, 16, 16, None) == -1
    assert lib.wr_push_shard_dma(None, 100, 2, 0, 16, None) == -1
    assert lib.wr_push_shard_dma(16, 100, 9, 0, 16, None) == -2
    assert lib.wr_push_marked_rows(None, 64, 16, 16, None) == -1
    shards = _lib.ShardsStruct()
    shards.world, shards.rank, shards.n_users, shards.n_items, shards.rows_u_local, shards.rows_i_local = 2, 0, 10, 7, 5, 4
    assert lib.wr_push_marked_rows(ctypes.addressof(shards), 64, 16, 16, None) == -1                     # bases not mapped
    assert lib.wr_csr_spmm_sharded_dma(16, 16, 16, 9, 64, None, 16, None, 0, None, None, 1.0, None, 16, 16, 64, 32, 1, 0, 16,
                                       None) == -1
    assert lib.wr_gather_rows_sharded(ctypes.addressof(shards), 0, 16, 4, 64, 16, 16, None) == -1        # bases not mapped
    shards.rows_u_local = 6
    assert lib.wr_gather_rows_sharded(ctypes.addressof(shards), 0, 16, 4, 64, 16, 16, None) == -2        # layout mismatch


def test_unsupported_embedding_size_is_refused_at_construction():
    """Sizes the evaluation kernels do not cover fail when the model is built, not after the first epoch."""
    corpus = ml100k_corpus()
    for cls in (BPRMF, LightGCN):
        with pytest.raises(ValueError, match='embedding_size'):
            cls(model_args(cls, embedding_size=96), corpus)
    assert BPRMF(model_args(BPRMF, embedding_size=128), corpus).emb_size == 128


def test_product_refuses_cpu_tensors():
    with pytest.raises(_lib.WhisprError):
        _lib.ptr(torch.zeros(4))
    corpus = ml100k_corpus()
    model = BPRMF(model_args(BPRMF), corpus)
    with pytest.raises(_lib.WhisprError):
        model.fuse()                                   # parameters still on the CPU: no fallback


def test_negative_sampler_bit_exact_on_ml100k():
    """Dataset.actions_before_epoch == reference BaseModel.py:167-177 on NumPy's global stream."""
    g = load('ml100k_bprmf.npz')
    corpus = ml100k_corpus()
    utils.init_seed(3407)
    model = BPRMF(model_args(BPRMF), corpus)
    ds = BPRMF.Dataset(model, corpus, 'train')
    ds.actions_before_epoch()
    assert ds.data['neg_items'].dtype == np.int64
    assert (ds.data['neg_items'] == g['neg_epoch1']).all()
    ds.actions_before_epoch()
    assert hashlib.sha256(ds.data['neg_items'].astype(np.int64).tobytes()).hexdigest() == str(g['neg_epoch2_sha'])
    assert (ds.data['neg_items'][:64] == g['neg_epoch2_head']).all()


def test_init_and_batch_order_bit_exact_on_ml100k():
    g = load('ml100k_bprmf.npz')
    corpus = ml100k_corpus()
    utils.init_seed(3407)
    model = BPRMF(model_args(BPRMF), corpus)
    assert hashlib.sha256(model.user_embeddings.weight.detach().numpy().tobytes()).hexdigest() == str(g['init_user_sha'])
    assert hashlib.sha256(model.item_embeddings.weight.detach().numpy().tobytes()).hexdigest() == str(g['init_item_sha'])
    assert model.count_variables() == 161088
    assert sorted(model.state_dict().keys()) == ['item_embeddings.weight', 'user_embeddings.weight']
    ds = BPRMF.Dataset(model, corpus, 'train')
    ds.actions_before_epoch()
    perm = dataloader_draws(len(ds), shuffle=True)
    for b in (0, 1):
        sel = perm[b * 2048:(b + 1) * 2048]
        assert (ds.data['user_id'][sel] == g[f'batch{b}_user']).all()
        assert (ds.data['item_id'][sel] == g[f'batch{b}_pos']).all()
        assert (ds.data['neg_items'][sel] == g[f'batch{b}_neg']).all()


def test_dataloader_draws_match_a_real_dataloader():
    from torch.utils.data import DataLoader
    for shuffle in (True, False):
        torch.manual_seed(5)
        dl = DataLoader(list(range(1000)), batch_size=64, shuffle=shuffle)
        ref = torch.cat([b for b in dl]).numpy()
        after_ref = torch.empty((), dtype=torch.int64).random_().item()
        torch.manual_seed(5)
        perm = dataloader_draws(1000, shuffle)
        after = torch.empty((), dtype=torch.int64).random_().item()
        assert after == after_ref                      # the global generator is left in the same state
        assert (ref == (perm if shuffle else np.arange(1000))).all()


def test_lightgcn_init_and_adjacency_structure():
    g = load('ml100k_lightgcn.npz')
    corpus = ml100k_corpus()
    utils.init_seed(3407)
    model = LightGCN(model_args(LightGCN, lr=2e-3), corpus)
    assert hashlib.sha256(model.user_embedding.weight.detach().numpy().tobytes()).hexdigest() == str(g['init_user_sha'])
    assert hashlib.sha256(model.item_embedding.weight.detach().numpy().tobytes()).hexdigest() == str(g['init_item_sha'])
    assert sorted(model.state_dict().keys()) == ['item_embedding.weight', 'user_embedding.weight']
    rowptr, col, dinv = model._adj_host
    c = load('ml100k_corpus.npz')
    o_rowptr, o_col, o_val = O.build_norm_adj_csr(c['n_users'], c['n_items'], c['train_user'], c['train_item'])
    assert (rowptr == o_rowptr).all() and (col == o_col).all()
    rows = np.repeat(np.arange(len(rowptr) - 1), np.diff(rowptr))
    val = (dinv[rows] * np.float32(1.0)) * dinv[col]            # what wr_csr_norm_weights computes
    assert val.dtype == np.float32 and val.tobytes() == o_val.tobytes()
    assert hashlib.sha256(val.tobytes()).hexdigest() == str(g['adj_val_sha'])


def test_history_csr_matches_oracle():
    corpus = ml100k_corpus()
    c = load('ml100k_corpus.npz')
    tr = np.stack([c['train_user'], c['train_item']], 1).astype(np.int64)
    rest = np.concatenate([np.stack([c['dev_user'], c['dev_item']], 1), np.stack([c['test_user'], c['test_item']], 1)])
    op, oi = O.history_csr(int(c['n_users']), tr, rest.astype(np.int64))
    hp, hi = corpus.history_csr()
    assert (hp == op).all() and (hi == oi).all()
    for u in (0, 17, 942):
        assert set(hi[hp[u]:hp[u + 1]]) == corpus.train_clicked_set[u] | corpus.residual_clicked_set[u]


def test_reader_reproduces_reference_split(tmp_path):
    """The reader's filter, id remap and seeded 80/10/10 split reproduce the reference's ml-100k split
    (tests/golden/ml100k_corpus.npz).  The input `.inter` is rebuilt from that split: its rows go back to file order by
    inverting the two seeded shuffles, and raw ids are a seeded permutation of the codes, so only a remap by first
    appearance gives the codes back.  Kept rows are rated 3 to 5 (3 is the floor).  Users left with fewer than 20 rows are
    padded with ratings 1 and 2, which the reader counts for the user filter and then drops.  One more user has 19
    above-floor rows and must be filtered out."""
    from sklearn.model_selection import train_test_split
    c = load('ml100k_corpus.npz')
    parts = [np.stack([c[ph + '_user'], c[ph + '_item']], 1).astype(np.int64) for ph in ('train', 'dev', 'test')]
    n = sum(len(p) for p in parts)
    train_at, rest_at = train_test_split(np.arange(n), train_size=0.8, random_state=42, shuffle=True)
    dev_at, test_at = train_test_split(rest_at, train_size=0.5, random_state=42, shuffle=True)
    rows = np.empty((n, 2), dtype=np.int64)
    for at, p in zip((train_at, dev_at, test_at), parts):
        rows[at] = p
    cnt = np.bincount(rows[:, 0])
    short = np.nonzero(cnt < 20)[0]
    assert len(short) > 0
    pad = np.repeat(short, 20 - cnt[short])
    rng = np.random.RandomState(5)
    user_token = rng.permutation(int(c['n_users'])) + 1
    item_token = rng.permutation(int(c['n_items'])) + 1
    users = np.concatenate([user_token[rows[:, 0]], user_token[pad], np.full(19, 5000)])
    items = np.concatenate([item_token[rows[:, 1]], np.full(len(pad) + 19, item_token[0])])
    rating = np.concatenate([rng.randint(3, 6, n), rng.randint(1, 3, len(pad)), np.full(19, 5)])
    assert (rating[:n] == 3).any() and (rating[n:n + len(pad)] == 2).any()
    inter = pd.DataFrame({'user_id:token': users, 'item_id:token': items, 'rating:float': rating,
                          'timestamp:float': 874_724_710 + np.arange(len(users))})
    os.makedirs(tmp_path / 'ml-100k')
    inter.to_csv(tmp_path / 'ml-100k' / 'ml-100k.inter', sep='\t', index=False)
    corpus = BaseReader(model_args(BPRMF, path=str(tmp_path), dataset='ml-100k'))
    assert int(corpus.n_users) == int(c['n_users']) == 943 and int(corpus.n_items) == int(c['n_items']) == 1574
    for ph in ('train', 'dev', 'test'):
        assert (corpus.data_df[ph]['user_id'].to_numpy() == c[ph + '_user']).all()
        assert (corpus.data_df[ph]['item_id'].to_numpy() == c[ph + '_item']).all()


def test_cli_surface_matches_reference():
    init_args, args, (model_class, reader_class, runner_class, reader_name) = wr_main.build_args(
        ['--model_name', 'LightGCN', '--emb_size', '32', '--gcn_layers', '3', '--lr', '2e-3', '--bogus', '1'])
    assert model_class is LightGCN and reader_name == 'BaseReader' and runner_class is BaseRunner
    assert args.embedding_size == 64                   # `--emb_size` is silently ignored, as in the reference
    assert args.gcn_layers == 3 and args.lr == 2e-3 and args.batch_size == 2048 and args.topk == '10,20'
    assert args.log_file == '../log/LightGCN/LightGCN__ml-100k__3407__lr=0.002__l2=0__embedding_size=64__' \
                            'gcn_layers=3__reg_weight=1e-05.txt'
    assert args.model_path.endswith('.pt') and '/model/LightGCN/' in args.model_path
    with pytest.raises(NameError):
        wr_main.build_args(['--model_name', 'NoSuchModel'])


def test_metric_formatting_and_host_metrics():
    res = {'NDCG@10': np.float64(0.05551), 'HR@10': np.float64(0.1087), 'HR@20': 0.25, 'NDCG@20': np.float32(0.1)}
    assert utils.format_metric(res) == 'HR@10:0.1087,NDCG@10:0.0555,HR@20:0.2500,NDCG@20:0.1000'
    s = load('small_cases.npz')
    pred, rank = s['bprmf_d16/eval_pred'], s['bprmf_d16/eval_rank']
    out = BaseRunner.evaluate_method(pred, [5, 10, 20], ['NDCG', 'HR', 'RECALL', 'PRECISION'])
    for k, v in zip(s['bprmf_d16/eval_keys'], s['bprmf_d16/eval_vals']):
        assert out[str(k)] == pytest.approx(float(v), rel=1e-12)
    assert BaseRunner.metrics_from_ranks(rank, [10], ['HR'])['HR@10'] == out['HR@10']
    with pytest.raises(ValueError):
        BaseRunner.metrics_from_ranks(rank, [10], ['MAP'])


def test_early_stop_rule():
    r = BaseRunner(model_args(BPRMF))
    assert not r.eval_termination([0.1] * 5)
    assert r.eval_termination([0.5] + [0.4] * 10)                  # best is more than early_stop epochs old
    assert r.eval_termination(list(np.linspace(1.0, 0.0, 11)))     # non-increasing for early_stop epochs


def test_spmm_plan_slices_tile_the_long_rows_exactly():
    rng = np.random.RandomState(1)
    deg = rng.poisson(20, size=500)
    deg[[3, 77, 400]] = [129, 1000, 4097]
    rowptr = np.zeros(501, dtype=np.int64)
    np.cumsum(deg, out=rowptr[1:])
    plan = _lib.SpmmPlan(rowptr, 64, 'cpu', threshold=128, chunk=128)
    assert plan.n_long == 3 and plan.n_chunks == 2 + 8 + 33
    row, beg, ln, slot = (x.numpy() for x in (plan.chunk_row, plan.chunk_beg, plan.chunk_len, plan.chunk_slot))
    assert (plan.slot_chunks.numpy() == [2, 8, 33]).all()
    for s, r in enumerate([3, 77, 400]):
        sel = slot == s
        assert (row[sel] == r).all()
        assert beg[sel][0] == rowptr[r] and (beg[sel][1:] == beg[sel][:-1] + ln[sel][:-1]).all()
        assert beg[sel][-1] + ln[sel][-1] == rowptr[r + 1] and ln[sel].max() <= 128 and ln[sel].min() >= 1
    assert _lib.SpmmPlan(rowptr, 64, 'cpu', threshold=10_000).ref() is None      # nothing to split


def test_bench_reference_arm_prints_one_contract_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm of the benchmark): exactly one JSON line on stdout with the contract
    keys, nothing else there; --dump-outputs writes the last step's loss and tables as float32 .npy files."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = tmp_path / 'outputs'
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '3', '--dump-outputs', str(dump)], capture_output=True, text=True, timeout=900,
                       cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'train_interactions_per_s' and d['unit'] == 'interactions/s'
    assert d['higher_is_better'] is True and d['value'] > 0 and d['n_gpus'] == 1
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config']
    out = {f: np.load(dump / f) for f in os.listdir(dump)}
    assert sorted(out) == ['item_embeddings.npy', 'loss.npy', 'user_embeddings.npy']
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in out.values())
    assert out['loss.npy'].shape == (1,) and out['user_embeddings.npy'].shape == (6040, 64)
    assert out['item_embeddings.npy'].shape == (3706, 64)
    # the tables after the timed steps, not the seeded initial ones; Adam moves a parameter by about lr per step
    import bench
    from whisprrec_b200.utils import synthetic
    U0, I0, _ = bench.cpu_problem(synthetic.ml1m_shaped_corpus(cache_dir=os.path.join(bench.CACHE, 'ref')))
    n_steps = 3 * 5 + 1 * 100                          # warmup * 5 + steps * 100 batches (run_reference)
    for got, init in ((out['user_embeddings.npy'], U0.numpy()), (out['item_embeddings.npy'], I0.numpy())):
        moved = np.abs(got - init).max()
        assert 0.1 * bench.LR < moved <= 2 * bench.LR * n_steps, moved
    assert 0.0 < out['loss.npy'][0] < np.log(2.0)      # BPR starts at log 2 on these near-zero tables and falls


@pytest.mark.parametrize('n,k', [(10, 3), (10, 10), (21, 6), (22, 6), (100, 90), (1000, 5), (100000, 7), (200000, 180000),
                                 (1 << 33, 4), (0, 0)])
def test_library_replica_of_python_random_sample(n, k):
    """wr_pyrandom_sample (host code in the library) == random.sample(range(n), k), including the generator state it
    leaves behind -- both branches of CPython's algorithm (pool shuffle / set of picks) and ranges beyond 32 bits.
    SGL's per-epoch edge dropout (reference utils/augmentor.py:77-111) is this call."""
    import random
    random.seed(3407)
    random.random()                                    # not at a block boundary
    want = random.sample(range(n), k)
    after = random.random()
    random.seed(3407)
    random.random()
    got = _lib.py_random_sample(n, k)
    assert got.tolist() == want
    assert random.random() == after


@pytest.mark.parametrize('tag', ['sgl_d16_l2', 'sgl_d32_l3'])
def test_sgl_edge_dropout_views_match_reference(tag):
    """The two augmented views of an epoch, built from our CSR with the library's replica of Python's random stream,
    equal the reference's sub-graphs bit for bit (tests/golden/sgl_cases.npz)."""
    import random
    from tests.helpers import load, small_case
    from whisprrec_b200.models.general.LightGCN import build_norm_adj_csr
    from whisprrec_b200.utils.graph_views import edge_dropout_view
    s = small_case(load('sgl_cases.npz'), tag)
    nU, nI, drop = s['U0'].shape[0], s['I0'].shape[0], float(s['hp'][7])
    N = nU + nI
    tr = np.unique(s['train'].astype(np.int64), axis=0)
    ptr = np.zeros(nU + 1, dtype=np.int64)
    np.cumsum(np.bincount(tr[:, 0], minlength=nU), out=ptr[1:])
    rowptr, col, _ = build_norm_adj_csr(nU, nI, ptr, tr[:, 1].astype(np.int32))
    random.seed(1234)
    def dense_of(vp, vc, vv):
        d = np.zeros((N, N), dtype=np.float32)
        d[np.repeat(np.arange(N), np.diff(vp)), vc] = vv
        return d
    for name in ('sub1', 'sub2'):
        fwd, tr_ = edge_dropout_view(rowptr, col, drop, transpose=True)
        assert (dense_of(*fwd) == s[name]).all(), name
        assert (dense_of(*tr_) == s[name].T).all(), name + ' transposed'        # what the adjoint propagation multiplies by


def test_sgl_model_keeps_the_reference_flags():
    """`--model_name SGL` resolves, and its flags / defaults / log arguments are the reference's (SGL.py:20-42)."""
    from whisprrec_b200.main import resolve
    cls = resolve('model', 'SGL')
    a = model_args(cls)
    assert (a.embedding_size, a.gcn_layers, a.type, a.reg_weight, a.ssl_tau, a.ssl_weight, a.drop_ratio) == \
        (64, 2, 'ED', 1e-4, 0.1, 0.05, 0.1)
    assert cls.extra_log_args == ['embedding_size', 'gcn_layers', 'reg_weight', 'type', 'ssl_tau', 'ssl_weight', 'drop_ratio']
    assert cls.reader == 'BaseReader' and cls.runner == 'BaseRunner'


def test_checkpoints_have_the_reference_state_dict_layout(tmp_path):
    """SURVEY.md section 8 f-4 without the reference checkout: the state_dict a `.pt` of ours holds has exactly the keys,
    shapes and dtypes of the unmodified reference's models (tests/golden/reference_state_dicts.json, written by
    tests/golden/make_golden_keys.py from the reference classes), and survives save / load (BaseModel.py:48-59)."""
    import json
    from tests.helpers import GOLDEN
    from whisprrec_b200.main import resolve
    want = json.load(open(os.path.join(GOLDEN, 'reference_state_dicts.json')))
    corpus = ml100k_corpus()
    for name, layout in want.items():
        cls = resolve('model', name)
        m = cls(model_args(cls), corpus)
        got = {k: [list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()}
        assert got == layout, name
        path = str(tmp_path / (name + '.pt'))
        torch.save(m.state_dict(), path)
        back = torch.load(path)
        assert list(back.keys()) == list(m.state_dict().keys())
        for k in back:
            assert torch.equal(back[k], m.state_dict()[k])


def test_corpus_cache_is_written_under_the_reference_class_path(tmp_path):
    """SURVEY.md section 8 f-4, both directions: the cache main.py writes names `helpers.BaseReader.BaseReader` (what the
    reference's `pickle.load` resolves to ITS reader class, main.py:54-63) and no module of this package; it loads back
    here as our reader with every attribute intact.  (The run against the real reference is the next test.)"""
    import pickle
    from whisprrec_b200 import main as wr_main
    from whisprrec_b200.helpers.BaseReader import BaseReader
    corpus = ml100k_corpus()
    pkl = str(tmp_path / 'BaseReader.pkl')
    wr_main.save_corpus(corpus, pkl)
    raw = open(pkl, 'rb').read()
    assert b'helpers.BaseReader' in raw and b'whisprrec_b200' not in raw
    assert 'helpers' not in __import__('sys').modules or not hasattr(__import__('sys').modules['helpers'], '__wr_alias__')
    back = wr_main.load_corpus(pkl)
    assert type(back) is BaseReader and (back.n_users, back.n_items) == (corpus.n_users, corpus.n_items)
    assert back.train_clicked_set == corpus.train_clicked_set and back.residual_clicked_set == corpus.residual_clicked_set
    for ph in ('train', 'dev', 'test'):
        assert back.data_df[ph].equals(corpus.data_df[ph])
    # a cache the reference wrote lacks `_csr_cache`, the one attribute only this package sets: the CSR views the
    # kernels consume are rebuilt on demand from the splits
    ref_like = BaseReader.__new__(BaseReader)
    ref_like.__dict__.update({k: v for k, v in corpus.__dict__.items() if k != '_csr_cache'})
    wr_main.save_corpus(ref_like, pkl)
    back = wr_main.load_corpus(pkl)
    assert type(back) is BaseReader and '_csr_cache' not in back.__dict__
    for view in ('train_csr', 'history_csr'):
        for a, b in zip(getattr(back, view)(), getattr(corpus, view)()):
            assert a.dtype == b.dtype and (a == b).all(), view

    class Theirs(object):                    # what the reference does: its own class, object.__new__ + __dict__
        pass

    class U(pickle.Unpickler):
        def find_class(self, module, name):
            if (module, name) == ('helpers.BaseReader', 'BaseReader'):
                return Theirs
            return super().find_class(module, name)
    with open(pkl, 'rb') as f:
        theirs = U(f).load()
    assert type(theirs) is Theirs and theirs.n_items == corpus.n_items and len(theirs.data_df['train']) == len(corpus.data_df['train'])


@needs_reference
def test_our_corpus_cache_loads_in_the_reference(tmp_path):
    """The same file through the reference's own code path: `pickle.load` in a process that has the reference's `src/` on
    its path (main.py:57-59) yields the reference's BaseReader with our ids and splits."""
    import subprocess
    import sys
    from whisprrec_b200 import main as wr_main
    corpus = ml100k_corpus()
    pkl = str(tmp_path / 'BaseReader.pkl')
    wr_main.save_corpus(corpus, pkl)
    code = f"""
import sys, pickle, numpy as np
np.float_ = np.float64
sys.path.insert(0, {REF_SRC!r})
from helpers.BaseReader import BaseReader
with open("{pkl}", "rb") as f:
    c = pickle.load(f)
assert type(c) is BaseReader, type(c)
print(c.n_users, c.n_items, len(c.data_df['train']), len(c.train_clicked_set))
"""
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split() == [str(corpus.n_users), str(corpus.n_items), str(len(corpus.data_df['train'])),
                                str(len(corpus.train_clicked_set))]


@needs_reference
def test_checkpoints_interchange_with_the_reference(tmp_path):
    """SURVEY.md section 8 f-4: a `.pt` written by the reference's BaseModel.save_model loads into ours and the other way
    round -- same state_dict keys, shapes, dtype (reference models/BaseModel.py:48-59)."""
    import subprocess
    import sys
    corpus = ml100k_corpus()
    ours = BPRMF(model_args(BPRMF), corpus)
    ours_path, ref_path = str(tmp_path / 'ours.pt'), str(tmp_path / 'ref.pt')
    torch.save(ours.state_dict(), ours_path)
    # the reference runs in its own interpreter: its top-level packages are called `models`, `helpers`, `utils`
    script = f'''
import sys, types, numpy as np, torch
np.float_ = np.float64
sys.path.insert(0, {REF_SRC!r})
from models.general.BPRMF import BPRMF
args = types.SimpleNamespace(device=torch.device("cpu"), model_path="", buffer=1, num_neg=1, test_all=1, embedding_size=64)
corpus = types.SimpleNamespace(n_users={int(corpus.n_users)}, n_items={int(corpus.n_items)})
m = BPRMF(args, corpus)
m.load_state_dict(torch.load("{ours_path}"))                      # ours -> reference, strict
torch.manual_seed(5)
m = BPRMF(args, corpus)
m.model_path = "{ref_path}"
m.save_model()                                                    # reference -> file
print("REF_SUM", float(m.user_embeddings.weight.double().sum()), float(m.item_embeddings.weight.double().sum()))
'''
    r = subprocess.run([sys.executable, '-c', script], capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    u_sum, i_sum = (float(x) for x in r.stdout.split('REF_SUM')[1].split())
    ours.load_state_dict(torch.load(ref_path))                        # reference -> ours, strict
    assert float(ours.user_embeddings.weight.double().sum()) == u_sum
    assert float(ours.item_embeddings.weight.double().sum()) == i_sum


@needs_reference
def test_reference_corpus_cache_loads_as_our_reader(tmp_path):
    """SURVEY.md section 8 f-4: a `BaseReader.pkl` cached by the reference (main.py:54-63) is picked up by `--regenerate 0`
    here: it unpickles as this package's reader and yields the same splits and CSR views."""
    import subprocess
    import sys
    from whisprrec_b200 import main as wr_main
    pkl = str(tmp_path / 'BaseReader.pkl')
    script = f'''
import sys, types, pickle, numpy as np
np.float_ = np.float64
sys.path.insert(0, {REF_SRC!r})
from helpers.BaseReader import BaseReader
args = types.SimpleNamespace(sep="\\t", path={REF_DATA!r}, dataset="ml-100k", sample="random")
with open("{pkl}", "wb") as f:
    pickle.dump(BaseReader(args), f)
'''
    r = subprocess.run([sys.executable, '-c', script], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    theirs = wr_main.load_corpus(pkl)
    from whisprrec_b200.helpers.BaseReader import BaseReader
    assert type(theirs) is BaseReader
    mine = ml100k_corpus()
    assert int(theirs.n_users) == int(mine.n_users) and int(theirs.n_items) == int(mine.n_items)
    for ph in ('train', 'dev', 'test'):
        assert (theirs.data_df[ph]['user_id'].to_numpy() == mine.data_df[ph]['user_id'].to_numpy()).all()
        assert (theirs.data_df[ph]['item_id'].to_numpy() == mine.data_df[ph]['item_id'].to_numpy()).all()
    for a, b in zip(theirs.history_csr(), mine.history_csr()):
        assert (a == b).all()
    for a, b in zip(theirs.train_csr(), mine.train_csr()):
        assert (a == b).all()
