#!/bin/bash
# Round-end ncu evidence, run on the GPU box through gpurun (one GPU).  The .ncu-rep files stay in /tmp on the box
# (they exceed gpurun's 64 MiB return limit); CSV exports come back in gpurun_out/.  Every command runs once
# without ncu first.
#   gpurun --timeout 1700 -- 'bash tools/capture_profiles.sh r2a'
set -u
TAG=${1:-r2x}
OUT=gpurun_out
B="python bench.py --steps 20 --warmup 5 --no-e2e --no-cpu --no-secondary"
full() {  # full <name> <kernel regex> <skip> <count> <command...>
    local name=$1 rx=$2 skip=$3 cnt=$4; shift 4
    "$@" > $OUT/plain_${TAG}_${name}.log 2>&1 || { echo "plain run of $name failed"; tail -3 $OUT/plain_${TAG}_${name}.log; return; }
    ncu --set full --clock-control none --import-source on -k regex:$rx --launch-skip $skip --launch-count $cnt \
        -o /tmp/prof_${TAG}_${name} -f "$@" > $OUT/ncu_${TAG}_${name}.log 2>&1
    ncu -i /tmp/prof_${TAG}_${name}.ncu-rep --page raw --csv > $OUT/full_${TAG}_${name}.csv 2>/dev/null
}
$B > $OUT/plain_${TAG}.log 2>&1 || { echo "plain bench failed"; tail -5 $OUT/plain_${TAG}.log; exit 1; }
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches_${TAG}.csv $B > $OUT/ncu1_${TAG}.log 2>&1
full step  hk_sched_kernel 21 21 python tools/time_census.py c2 2 census
full c5    "hk_(rows|generic)_kernel" 42 42 python tools/time_census.py c5 2 census
full obs   hk_small_kernel 41 20 python tools/profile_misc.py obs_c2
full rollc2 hk_small_kernel 3 1 python tools/profile_misc.py rollout_c2
full rollc5 hk_generic_kernel 3 1 python tools/profile_misc.py rollout_c5
tail -1 $OUT/plain_${TAG}.log | cut -c1-300; ls $OUT | grep ${TAG}
