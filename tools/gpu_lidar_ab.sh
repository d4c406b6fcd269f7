#!/bin/bash
# k_lidar A/B: the in-tree library and every variants/*.so on the config-2 / config-4 shapes.  usage: bash tools/gpu_lidar_ab.sh tag
TAG=${1:-lab}; OUT=gpurun_out/$TAG; mkdir -p $OUT
for rep in 1 2; do
  for spec in austria:4096 treitlstrasse_v2:65536 columbia:16384; do
    echo "== base $spec" | tee -a $OUT/ab.log; RD_SWEEP=$spec python tools/lidar_sweep.py 2>&1 | tail -1 | tee -a $OUT/ab.log
    for v in variants/*.so; do
      [ -f "$v" ] || continue
      echo "== $(basename $v .so) $spec" | tee -a $OUT/ab.log; RD_ENV_LIB=$PWD/$v RD_SWEEP=$spec python tools/lidar_sweep.py 2>&1 | tail -1 | tee -a $OUT/ab.log
    done
  done
done
