#!/bin/bash
# Round-2 full pass in one gpurun call: parity suite (all failures listed), smoke, bench (product, reference, dense),
# batch phase clocks, ncu launch lists and --set full captures of the dominant kernels.  Logs go to gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
nproc > gpurun_out/nproc.txt
( time timeout 2400 python -m pytest tests -q -m gpu ) > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
( time timeout 300 python -c "import __graft_entry__ as g; g.smoke()" ) > gpurun_out/smoke.log 2>&1
( time timeout 1200 python bench.py --steps 5 --warmup 3 ) > gpurun_out/bench.log 2>&1
( time timeout 600 python bench.py --impl reference --steps 2 --warmup 1 ) > gpurun_out/bench_ref.log 2>&1
( time timeout 900 python bench.py --workload dense --steps 2 --warmup 3 ) > gpurun_out/bench_dense.log 2>&1
python tools/batch_phases.py 512 > gpurun_out/batch_phases.txt 2>&1
python tools/prof_dense.py 8000 potrf_prof > gpurun_out/potrf_prof.txt 2>&1
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 6000 --csv --log-file gpurun_out/launches_batch.csv \
   python bench.py --steps 1 --warmup 1 --no-dense --no-cpu > gpurun_out/ncu_batch.log 2>&1
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 20000 --csv --log-file gpurun_out/launches_dense.csv \
   python bench.py --workload dense --steps 1 --warmup 1 --no-cpu > gpurun_out/ncu_dense.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:kbp_solve -s 1 -c 1 -f -o gpurun_out/full_kbp_solve \
   python bench.py --steps 1 --warmup 1 --no-dense --no-cpu > gpurun_out/ncu_full_batch.log 2>&1
tail -5 gpurun_out/pytest_gpu.log; tail -2 gpurun_out/smoke.log; tail -c 1500 gpurun_out/bench.log; tail -c 800 gpurun_out/bench_ref.log; tail -c 800 gpurun_out/bench_dense.log
ls -la gpurun_out
