#!/bin/bash
# End-of-round-2 pass in one gpurun call: parity suite, smoke, bench (product, reference, dense), batch phase clocks, update-path
# micro-benchmarks, sparse profile, ncu launch lists and --set full captures of the dominant kernels.  Logs go to gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
nproc > gpurun_out/nproc.txt
( time timeout 2400 python -m pytest tests -q -m gpu -rs ) > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
( time timeout 300 python -c "import __graft_entry__ as g; g.smoke()" ) > gpurun_out/smoke.log 2>&1
( time timeout 1200 python bench.py --steps 5 --warmup 3 ) > gpurun_out/bench.log 2>&1
( time timeout 600 python bench.py --impl reference --steps 2 --warmup 1 ) > gpurun_out/bench_ref.log 2>&1
( time timeout 900 python bench.py --workload dense --steps 3 --warmup 3 ) > gpurun_out/bench_dense.log 2>&1
python tools/batch_phases.py 512 > gpurun_out/batch_phases.txt 2>&1
( timeout 600 python tools/c3_trace.py ) > gpurun_out/c3_trace_gen.txt 2>&1
( timeout 300 python tools/prof_config.py c3; timeout 300 python tools/prof_config.py c1; timeout 300 python tools/prof_config.py c5 ) > gpurun_out/prof_c3_c1_c5.txt 2>&1
( QPALM_B200_MF_CLOCKS=1 timeout 600 python tools/prof_config.py grid300; QPALM_B200_MF_PER_BLOCK=1 timeout 600 python tools/prof_config.py grid300 | head -3 ) > gpurun_out/prof_grid300_cluster.txt 2>&1
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 6000 --csv --log-file gpurun_out/launches_batch.csv \
   python bench.py --steps 1 --warmup 1 --no-dense --no-cpu --sweep-total 0 > gpurun_out/ncu_batch.log 2>&1
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 12000 --csv --log-file gpurun_out/launches_dense.csv \
   python bench.py --workload dense --steps 1 --warmup 1 --no-cpu > gpurun_out/ncu_dense.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:kbp_solve -s 1 -c 1 -f -o gpurun_out/full_kbp_solve \
   python bench.py --steps 1 --warmup 1 --no-dense --no-cpu --sweep-total 0 > gpurun_out/ncu_full_batch.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_fwd_multi -s 40 -c 1 -f -o gpurun_out/full_k_fwd_multi \
   python tools/c3_trace.py > gpurun_out/ncu_full_fwd.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_gen_apply -s 40 -c 1 -f -o gpurun_out/full_k_gen_apply \
   python tools/c3_trace.py > gpurun_out/ncu_full_apply.log 2>&1
tail -8 gpurun_out/pytest_gpu.log; tail -2 gpurun_out/smoke.log; tail -c 2500 gpurun_out/bench.log; tail -c 800 gpurun_out/bench_ref.log; tail -c 1200 gpurun_out/bench_dense.log
ls -la gpurun_out | tail -30
