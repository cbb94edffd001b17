#!/bin/bash
# ncu --set full capture of selected kernels from one bench step (single GPU).
mkdir -p gpurun_out
TAG=${TAG:-r01}
timeout 900 ncu --set full --clock-control none --import-source on \
   -k regex:"${KERNELS:-app_basis_fwd_kernel|head_mlp_fwd_kernel|head_bwd_data_kernel|head_bwd_wgrad_kernel|vm_bwd_kernel|vm_fwd_kernel}" -s ${SKIP:-10} -c ${COUNT:-7} \
   -o gpurun_out/${TAG}_prof -f python bench.py --steps 1 --warmup 3 --no-cpu-baseline --no-breakdown ${BENCH_ARGS} > gpurun_out/${TAG}_prof.log 2>&1
ls -la gpurun_out | tail -8
