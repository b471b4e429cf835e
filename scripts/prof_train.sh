#!/bin/bash
# Training-step evidence: graph-replay time, per-phase event times,
# and the ncu launch list of one eager step (kernel shares).  Outputs under gpurun_out/.
set -u
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
python scripts/bench_train.py --steps 40 --warmup 5 --profile > gpurun_out/train_default.json 2> gpurun_out/train_default.err
tail -1 gpurun_out/train_default.json | cut -c1-600
ncu --metrics gpu__time_duration.sum --clock-control none -c 1200 --csv --log-file gpurun_out/train_launches_r02.csv \
  python scripts/bench_train.py --eager --steps 1 --warmup 2 > gpurun_out/ncu_train.log 2>&1
python scripts/agg_launches.py gpurun_out/train_launches_r02.csv --last 200 > gpurun_out/train_launches_r02_summary.txt 2>&1
head -50 gpurun_out/train_launches_r02_summary.txt
