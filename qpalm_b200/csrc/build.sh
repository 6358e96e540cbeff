#!/bin/bash
# Builds libqpalm_b200.so in-tree for sm_100a.  -fmad=false keeps element-wise arithmetic bit-identical to
# the reference's (non-FMA) C loops; hot dense loops use explicit fma()/DMMA.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -fmad=false $QB_EXTRA_FLAGS"
mkdir -p build
pids=()
for f in dense updown_gen kernels api ops compat kkt batch batchp prof shard sparse sparse_sym qps; do
  if [ ! -f build/$f.o ] || [ $f.cu -nt build/$f.o ] || [ engine.cuh -nt build/$f.o ] || [ dense.cuh -nt build/$f.o ] || [ common.cuh -nt build/$f.o ] || [ batch.cuh -nt build/$f.o ] || [ sparse.cuh -nt build/$f.o ] || [ sparse_host.h -nt build/$f.o ] || [ chol32.cuh -nt build/$f.o ] || [ ../../include/qpalm_b200.h -nt build/$f.o ]; then
    $NVCC $FLAGS -c $f.cu -o build/$f.o &
    pids+=($!)
  fi
done
# the persistent batch engine a second time in its 4-CTAs-per-SM shape (see the header of batchp.cu)
if [ ! -f build/batchp4.o ] || [ batchp.cu -nt build/batchp4.o ] || [ batch.cuh -nt build/batchp4.o ] || [ common.cuh -nt build/batchp4.o ] || [ engine.cuh -nt build/batchp4.o ]; then
  $NVCC $FLAGS -DQB_BP_VARIANT4 $QB_BP4_FLAGS -c batchp.cu -o build/batchp4.o &
  pids+=($!)
fi
# and both shapes once more with the test probes of its building blocks instead of the solver kernel (-DQB_BP_PROBE)
for v in batchp_probe batchp4_probe; do
  if [ ! -f build/$v.o ] || [ batchp.cu -nt build/$v.o ] || [ batch.cuh -nt build/$v.o ] || [ common.cuh -nt build/$v.o ] || [ engine.cuh -nt build/$v.o ] || [ chol32.cuh -nt build/$v.o ] || [ ../../include/qpalm_b200.h -nt build/$v.o ]; then
    if [ $v = batchp4_probe ]; then VF="-DQB_BP_VARIANT4 $QB_BP4_FLAGS"; else VF=""; fi
    $NVCC $FLAGS $VF -DQB_BP_PROBE -c batchp.cu -o build/$v.o &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -shared -o ../libqpalm_b200.so build/dense.o build/updown_gen.o build/kernels.o build/api.o build/ops.o build/compat.o build/kkt.o build/batch.o build/batchp.o build/batchp4.o build/batchp_probe.o build/batchp4_probe.o build/prof.o build/shard.o build/sparse.o build/sparse_sym.o build/qps.o -lcudart -ldl
echo "built $(cd .. && pwd)/libqpalm_b200.so"
