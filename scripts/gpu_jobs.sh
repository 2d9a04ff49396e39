#!/usr/bin/env bash
# The jobs this repo runs on a GPU box, one function each (run from the repo root: `bash scripts/gpu_jobs.sh <job>`).
# Every profiling job runs its command once without the profiler first; nothing here touches the GPU clocks.
set -u
cd "${GRAFT_REPO_ROOT:-$(dirname "$0")/..}"
mkdir -p gpurun_out

tests()      { timeout 1500 python -m pytest tests -x -q -m gpu 2>&1 | tail -6; }                         # 1 GPU
tests_dist() { timeout 900 python -m pytest tests/test_multi_gpu.py -x -q -m gpu 2>&1 | tail -4; }        # >= 2 GPUs
smoke()      { timeout 300 python __graft_entry__.py smoke 2>&1 | tail -3; }
bench1()     { timeout 900 python bench.py > gpurun_out/bench_n1.json 2> gpurun_out/bench_n1.err; echo "rc=$?"; }
benchN()     { # benchN 8
  timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node "$1" --master-addr 127.0.0.1 --master-port 29531 \
      bench.py --gpus "$1" > "gpurun_out/bench_n$1.json" 2> "gpurun_out/bench_n$1.err"; echo "rc=$?"; }
reference()  { timeout 400 python bench.py --impl reference --steps 20 --warmup 3 > gpurun_out/reference_arm.json; echo "rc=$?"; }
resident()   { timeout 300 python scripts/prof_resident.py gpurun_out/prof_resident.json; }               # both resident kernels, streaming
owner()      { timeout 200 python scripts/prof_owner.py gpurun_out/prof_owner.json; }                     # per-CTA phases, one-barrier kernel
sharded()    { # sharded 8 [bprmf|lightgcn|both]      (WR_SPMM_PUSH=dma selects the copy-engine SpMM push)
  timeout 1500 python -m torch.distributed.run --nnodes=1 --nproc-per-node "$1" --master-addr 127.0.0.1 --master-port 29517 \
      scripts/prof_sharded.py "gpurun_out/prof_sharded_n$1.json" "${2:-both}" 2>&1 | tail -70; }
push_overlap() { # push_overlap 8
  timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node "$1" --master-addr 127.0.0.1 --master-port 29518 \
      scripts/prof_push_overlap.py "gpurun_out/prof_push_overlap_n$1.json" 1.0 4 2>&1 | tail -20; }
sgl_sharded() { # sgl_sharded 8      (merges into profiles/r08_bench_sgl_sharded.json; run 1, 2, 4 and 8)
  timeout 2400 python -m torch.distributed.run --nnodes=1 --nproc-per-node "$1" --master-addr 127.0.0.1 --master-port 29533 \
      scripts/bench_sgl_sharded.py --out profiles/r08_bench_sgl_sharded.json 2>&1 | tail -8; }
ncu_all()    { bash scripts/_ncu1.sh; bash scripts/_ncu2.sh; }                                            # `ncu --set full` captures -> profiles/ via scripts/ncu_summary.py

"$@"
