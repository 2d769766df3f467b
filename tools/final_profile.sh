#!/bin/bash
# Round-end evidence on one B200: bench lines of every workload, CUPTI timeline, ncu launch list, and `ncu --set full`
# captures of the tensor-core / bandwidth kernels of ONE eager training step (tools/ncu_step.py).  Outputs in gpurun_out/.
set -u
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
for w in ${BENCH_WORKLOADS:-cond_grid sample vae cond_grid1024 cond256}; do
  python bench.py --workload $w --steps 30 --warmup 5 > gpurun_out/bench_final_$w.log 2>&1
  grep "^{" gpurun_out/bench_final_$w.log > gpurun_out/bench_final_$w.json
done
python tools/timeline.py > gpurun_out/timeline_final.log 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv --log-file gpurun_out/launches_final.csv \
    python tools/ncu_step.py > gpurun_out/ncu_launches_final.log 2>&1
cap() {  # kernel regex, launch count, file tag.  The .ncu-rep is reduced to its raw-page CSV on the box and deleted: gpurun
         # only brings back 64 MiB, one 54-launch report with sources is already 80 MB
  timeout 900 ncu --set full --clock-control none --profile-from-start off -k regex:$1 -c $2 -f \
      -o gpurun_out/ncu_full_$3 python tools/ncu_step.py > gpurun_out/ncu_full_$3.log 2>&1
  tail -1 gpurun_out/ncu_full_$3.log
  ncu -i gpurun_out/ncu_full_$3.ncu-rep --page raw --csv > gpurun_out/ncu_full_$3_raw.csv 2>/dev/null
  rm -f gpurun_out/ncu_full_$3.ncu-rep
}
cap conv_tc_kernel 54 conv_tc
cap wgrad_tc_kernel 8 wgrad_tc
cap conv3_halo_kernel 6 conv3_halo
cap convT_halo_kernel 3 convT_halo
cap wgrad3_halo_kernel 4 wgrad3_halo
cap adam_multi_kernel 1 adam_multi
cap "bn_" 6 bn
cap "elbo_|reparam_|patch_tma" 6 elbo_reparam_patch
du -sh gpurun_out; ls -la gpurun_out | head -40
