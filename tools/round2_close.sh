#!/bin/bash
# Round-2 closing run at HEAD: counter diag, the whole GPU suite, smoke, the driver's bench command, sanitizers on the counter,
# ncu launch lists + full captures (counter, pileup network).
set -u
mkdir -p gpurun_out
R=${1:-r2p}
timeout -k 10 120 python tools/plp_diag.py diag > gpurun_out/${R}_plp_diag.log 2>&1; tail -2 gpurun_out/${R}_plp_diag.log
timeout -k 10 100 python tools/plp_diag.py prof 1048576 12 2>&1 | tail -1 | tee gpurun_out/${R}_plp_prof.log
timeout -k 10 700 python -m pytest tests -m gpu -q --timeout=120 > gpurun_out/${R}_pytest.log 2>&1; tail -4 gpurun_out/${R}_pytest.log
timeout -k 10 150 python __graft_entry__.py smoke > gpurun_out/${R}_smoke.log 2>&1; tail -4 gpurun_out/${R}_smoke.log
timeout -k 10 480 python bench.py --gpus 1 --steps 20 --warmup 5 > gpurun_out/${R}_bench.json 2> gpurun_out/${R}_bench.err; tail -c 600 gpurun_out/${R}_bench.err
python tools/bench_summary.py gpurun_out/${R}_bench.json > gpurun_out/${R}_bench_summary.md 2>&1; head -10 gpurun_out/${R}_bench_summary.md; tail -3 gpurun_out/${R}_bench_summary.md
SAN=/usr/local/cuda/bin/compute-sanitizer
for tool in memcheck racecheck; do
  timeout -k 10 200 $SAN --tool $tool --print-limit 5 python tools/plp_diag.py diag > gpurun_out/${R}_san_plp_${tool}.log 2>&1
  echo "$tool [pileup counter] :: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|DIAG' gpurun_out/${R}_san_plp_${tool}.log | tr '\n' ' ')"
done
timeout -k 10 120 ncu --metrics gpu__time_duration.sum --clock-control none -c 40 --csv --log-file gpurun_out/${R}_launches_plp.csv \
    python tools/plp_diag.py prof 1048576 3 > gpurun_out/${R}_ncu_launch_plp.log 2>&1
timeout -k 10 180 ncu --set full --clock-control none --import-source on -k regex:"plp_count_tile" -s 1 -c 1 \
    -o gpurun_out/${R}_prof_plp python tools/plp_diag.py prof 1048576 3 > gpurun_out/${R}_ncu_full_plp.log 2>&1
B="python bench.py --steps 4 --warmup 3 --no-cpu-baseline --streams 1"
timeout -k 10 200 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${R}_launches_pileup.csv \
    $B --workloads pileup > gpurun_out/${R}_ncu_launch_p.log 2>&1
timeout -k 10 300 ncu --set full --clock-control none --import-source on -k regex:"lstm_tc_kernel|lstm_pair_kernel|lstm2x|proj2_kernel|tail_kernel|ingest_pileup" -s 20 -c 5 \
    -o gpurun_out/${R}_prof_pileup $B --workloads pileup > gpurun_out/${R}_ncu_full_p.log 2>&1
ls -la gpurun_out | grep ${R}_ | head -40
