#!/bin/bash
# compute-sanitizer memcheck + racecheck on the flag / queue based kernels (kbp_solve, flow::k_solve_flow)
mkdir -p gpurun_out
CS=/usr/local/cuda/bin/compute-sanitizer
for which in batch dense sparse; do
  for tool in memcheck racecheck; do
    log=gpurun_out/sanitizer_${tool}_${which}.txt
    ( timeout 600 $CS --tool $tool --print-limit 20 python tools/sanitize_case.py $which ) > $log 2>&1
    echo "exit $?" >> $log
    echo "== $tool $which"; grep -E "ERROR SUMMARY|RACECHECK SUMMARY|exit |^batch|^dense|^sparse" $log | tail -4
  done
done
