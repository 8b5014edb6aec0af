#!/bin/bash
# ncu evidence for the headline workload (run under gpurun, one GPU).  Usage: scripts/profile_c2.sh <tag>
# Environment is inherited by the benchmark processes.
set -u
TAG=${1:-r1}
CMD="python bench.py --workload c2 --steps 2 --warmup 3 --no-cpu --chains-per-mag 1000 --niter 100 --e2e-steps 1"
$CMD > gpurun_out/plain_$TAG.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 40 --csv --log-file gpurun_out/launches_$TAG.csv $CMD > gpurun_out/ncu_launches_$TAG.log 2>&1
$CMD > gpurun_out/plain2_$TAG.log 2>&1 &&
ncu --set full --clock-control none --import-source on -k regex:chain_kernel -s 3 -c 1 -o gpurun_out/prof_$TAG $CMD > gpurun_out/ncu_full_$TAG.log 2>&1
tail -3 gpurun_out/ncu_full_$TAG.log
