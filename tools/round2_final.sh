#!/bin/bash
# Round-2 closing evidence run: full GPU test suite, smoke, the driver's bench command, sanitizers (pair LSTM path, both convolution
# forms), ncu launch list + full capture of the pileup kernels, full capture of the pconv_impl = 1 convolutions.
set -u
mkdir -p gpurun_out
R=${1:-r2k}
timeout -k 10 300 python -m pytest tests/test_gpu_parity.py -m gpu -q -x --timeout=90 -k "tensor_core_kernels_match_reference or conv_taps" > gpurun_out/${R}_gate.log 2>&1
if [ $? -ne 0 ]; then echo "GATE FAILED"; tail -40 gpurun_out/${R}_gate.log; exit 1; fi
timeout -k 10 900 python -m pytest tests -m gpu -q --timeout=120 > gpurun_out/${R}_pytest.log 2>&1; tail -4 gpurun_out/${R}_pytest.log
timeout -k 10 120 python __graft_entry__.py smoke > gpurun_out/${R}_smoke.log 2>&1; tail -2 gpurun_out/${R}_smoke.log
timeout -k 10 600 python bench.py --gpus 1 --steps 20 --warmup 5 > gpurun_out/${R}_bench.json 2> gpurun_out/${R}_bench.err; tail -c 400 gpurun_out/${R}_bench.err
python tools/bench_summary.py gpurun_out/${R}_bench.json > gpurun_out/${R}_bench_summary.md 2>&1; head -12 gpurun_out/${R}_bench_summary.md
SAN=/usr/local/cuda/bin/compute-sanitizer
for tool in memcheck racecheck synccheck; do
  timeout -k 10 300 $SAN --tool $tool --print-limit 5 python tools/sanitize_case.py p 256 lstm_tile=64 > gpurun_out/${R}_san_pairdefault_${tool}.log 2>&1
  echo "$tool [default pileup path, pair LSTM2] :: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|ok \(' gpurun_out/${R}_san_pairdefault_${tool}.log | tr '\n' ' ')"
  timeout -k 10 300 $SAN --tool $tool --print-limit 5 python tools/sanitize_case.py p 256 lstm1_impl=1 > gpurun_out/${R}_san_pair12_${tool}.log 2>&1
  echo "$tool [pair LSTM1 + LSTM2] :: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|ok \(' gpurun_out/${R}_san_pair12_${tool}.log | tr '\n' ' ')"
  timeout -k 10 300 $SAN --tool $tool --print-limit 5 python tools/sanitize_case.py f 16 > gpurun_out/${R}_san_fa_${tool}.log 2>&1
  echo "$tool [full-alignment] :: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|ok \(' gpurun_out/${R}_san_fa_${tool}.log | tr '\n' ' ')"
  timeout -k 10 300 $SAN --tool $tool --print-limit 5 python tools/sanitize_case.py f 16 pconv_impl=1 > gpurun_out/${R}_san_fa2_${tool}.log 2>&1
  echo "$tool [full-alignment, pconv_impl=1 (CTA pairs)] :: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|ok \(' gpurun_out/${R}_san_fa2_${tool}.log | tr '\n' ' ')"
done
B="python bench.py --steps 4 --warmup 3 --no-cpu-baseline --streams 1"
timeout -k 10 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${R}_launches_pileup.csv \
    $B --workloads pileup > gpurun_out/${R}_ncu_launch_p.log 2>&1
timeout -k 10 600 ncu --set full --clock-control none --import-source on -k regex:"lstm_tc_kernel|lstm_pair_kernel|proj2_kernel|tail_kernel|ingest_pileup" -s 20 -c 5 \
    -o gpurun_out/${R}_prof_pileup $B --workloads pileup > gpurun_out/${R}_ncu_full_p.log 2>&1
timeout -k 10 400 ncu --set full --clock-control none --import-source on -k regex:"pconv_kernel" -s 9 -c 9 \
    -o gpurun_out/${R}_prof_fa_pconv2 python tools/sanitize_case.py f 256 pconv_impl=1 reps=3 > gpurun_out/${R}_ncu_full_f2.log 2>&1
ls -la gpurun_out | grep ${R}_ | head -40
