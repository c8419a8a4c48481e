#!/bin/bash
# Round-2 ncu evidence (run under gpurun, one GPU): launch lists (kernel shares) and one `--set full` capture of every distinct
# kernel of both networks, single stream, every timed region exactly the K steps.
set -u
R=${1:-r2p}
mkdir -p gpurun_out
B="python bench.py --steps 4 --warmup 3 --no-cpu-baseline --streams 1"
timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${R}_launches_pileup.csv \
    $B --workloads pileup > gpurun_out/${R}_ncu_launch_p.log 2>&1
timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file gpurun_out/${R}_launches_fa.csv \
    $B --workloads fa > gpurun_out/${R}_ncu_launch_f.log 2>&1
# full captures: skip the first forwards (parity check, allocation passes), take one forward's worth of kernels
timeout 600 ncu --set full --clock-control none --import-source on -k regex:"lstm_tc_kernel|lstm_pair_kernel|proj2_kernel|tail_kernel|ingest_pileup" -s 20 -c 5 \
    -o gpurun_out/${R}_prof_pileup $B --workloads pileup > gpurun_out/${R}_ncu_full_p.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:"pconv_kernel|tail_kernel|spp_tc_kernel|ingest_fa" -s 48 -c 12 \
    -o gpurun_out/${R}_prof_fa $B --workloads fa > gpurun_out/${R}_ncu_full_f.log 2>&1
ls -la gpurun_out | grep ${R}_ | head -20
