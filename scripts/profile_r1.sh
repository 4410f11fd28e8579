#!/bin/bash
# Round-1 ncu evidence (run under gpurun, 1 GPU).  Reduced memory footprints (ncu saves/restores device memory between
# replay passes), same kernels and shapes as the default bench.
set -x
B="python bench.py --steps 20 --warmup 3 --vi-batch 256 --c5-states 16384 --cpu-seconds 1"
$B > gpurun_out/prof_plain.log 2>&1 || exit 1
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file gpurun_out/launches_r1b.csv $B > gpurun_out/ncu_l.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:backup_kernel -s 5 -c 1 -o gpurun_out/prof_r1b_backup_c4 $B --workload vi > gpurun_out/ncu_b.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:backup_kernel -s 5 -c 1 -o gpurun_out/prof_r1b_backup_c5 $B --workload c5 > gpurun_out/ncu_c.log 2>&1
I="python scripts/one_instance.py MiniGridRoomsContinuous.ergo1 SimpleGridEpisodic.comm3"
$I > gpurun_out/prof_plain2.log 2>&1 || exit 1
ncu --set full --clock-control none --import-source on -k regex:"sparse_hitting|sparse_vi_kernel|sparse_episodic" -c 3 -o gpurun_out/prof_r1b_sparse $I > gpurun_out/ncu_sp.log 2>&1
