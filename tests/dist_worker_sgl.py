#!/usr/bin/env python
"""Worker for tests/test_multi_gpu_sgl.py: row-sharded SGL, one B200 per rank.

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29566 tests/dist_worker_sgl.py

The checks of tests/test_sgl_sharded.py on real peer memory: three steps of both sgl_cases.npz tags through
model.shard() against the goldens (views, loss, gradients, parameters), then one ml-100k epoch and a dev evaluation
against the single-GPU epoch with the same seeds.
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from tests import test_sgl_sharded as T
    from whisprrec_b200 import sharded as S
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    world = dist.get_world_size()
    assert torch.cuda.device_count() >= world, 'one GPU per rank (never share a GPU between spinning ranks)'
    T.DEV = dev
    for tag in ('sgl_d16_l2', 'sgl_d32_l3'):
        T.golden_steps_body(tag, S.PeerGroup(dev))
    T.ml100k_epoch_body(S.PeerGroup(dev))
    print('dist_worker_sgl ok', flush=True)
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
