"""Item-sharded top-k lists of 100 items on two B200s (tests/dist_worker_topk_long.py); skips on fewer GPUs."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, 'tests', 'dist_worker_topk_long.py')


@pytest.mark.gpu
def test_sharded_long_topk_on_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs one GPU per rank (ranks that spin on each other must never share a GPU)')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29564', WORKER]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS='1'),
                       cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count('dist_worker_topk_long ok') == 2
