#!/bin/bash
# ncu captures of the kernels of the VO step (run under gpurun, one GPU): full sets of the top kernels + the launch list.
# usage: tools/ncu_vo.sh <tag>
set -u
tag=${1:-r2}
mkdir -p gpurun_out
cmd="python bench.py --steps 3 --warmup 3 --no-secondary --vo-threads 2"
for k in local_ba2_kernel pose_only_kernel sparse_align_kernel track_project_kernel; do
  timeout 400 ncu --set full --clock-control none --import-source on -k regex:$k -s 6 -c 2 -f -o gpurun_out/${tag}_$k $cmd > gpurun_out/${tag}_ncu_$k.log 2>&1
done
timeout 300 ncu --set full --clock-control none --import-source on -k regex:klt -s 1 -c 2 -f -o gpurun_out/${tag}_klt_kernel python tools/klt_tail.py > gpurun_out/${tag}_ncu_klt.log 2>&1
timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 6000 --csv --log-file gpurun_out/${tag}_launches.csv $cmd > gpurun_out/${tag}_launches.log 2>&1
