#!/bin/bash
# A/B timing of prebuilt library variants (variants/*.so): k_lidar / k_step per-launch times on the bench workload
OUT=gpurun_out/${1:-var}; mkdir -p $OUT
for rep in 1 2 3; do
  for v in variants/*.so; do
    echo -n "$v " | tee -a $OUT/variants.log
    RD_ENV_LIB=$PWD/$v RD_SWEEP=${2:-austria:4096} python tools/lidar_sweep.py 2>&1 | tail -1 | tee -a $OUT/variants.log
  done
done
