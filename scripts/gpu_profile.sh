#!/bin/bash
# ncu evidence: (1) launch list of a short bench run, (2) full capture of the heaviest kernels.
mkdir -p gpurun_out
TAG=${TAG:-r01}
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -s 400 -c 200 --csv \
   --log-file gpurun_out/${TAG}_launches.csv python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-breakdown > gpurun_out/${TAG}_bench_under_ncu.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on \
   -k regex:"${KERNELS:-app_basis_fwd_kernel|head_mlp_fwd_kernel|head_bwd_data_kernel|head_bwd_wgrad_kernel|vm_bwd_kernel|vm_fwd_kernel}" -s 10 -c ${COUNT:-7} \
   -o gpurun_out/${TAG}_prof -f python bench.py --steps 1 --warmup 3 --no-cpu-baseline --no-breakdown > gpurun_out/${TAG}_prof.log 2>&1
ls -la gpurun_out | tail -8
