#!/bin/bash
# Run on a 2+-GPU box (gpurun --gpus N): GPU tests incl. the NCCL ones, 1-GPU and N-GPU bench.
# Usage: tools/gpu_multi.sh <tag> <ngpus> [steps]
TAG=${1:-r1}
N=${2:-2}
STEPS=${3:-5}
OUT=gpurun_out
mkdir -p $OUT
python -W ignore -m pytest tests -x -q -m gpu 2>&1 | tail -8 | tee $OUT/pytest_gpu_$TAG.log
python bench.py --steps $STEPS --warmup 3 --no-cpu > $OUT/bench_${TAG}_g1.json 2> $OUT/bench_${TAG}_g1.err
tail -c 1500 $OUT/bench_${TAG}_g1.json; tail -3 $OUT/bench_${TAG}_g1.err
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29531 \
    bench.py --gpus $N --steps $STEPS --warmup 3 > $OUT/bench_${TAG}_g$N.json 2> $OUT/bench_${TAG}_g$N.err
tail -c 1500 $OUT/bench_${TAG}_g$N.json; tail -5 $OUT/bench_${TAG}_g$N.err
