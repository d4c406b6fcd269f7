#!/bin/bash
# k_lidar beam groups per work item (variants/gpi*.so).  usage: bash tools/gpu_lidar_gpi.sh tag
TAG=${1:-gpi}; OUT=gpurun_out/$TAG; mkdir -p $OUT
for v in variants/gpi*.so; do
  echo "== tests $v"; RD_ENV_LIB=$PWD/$v timeout 600 python -m pytest tests/test_gpu_parity.py -x -q -m gpu -k "lidar or closed_loop or mixed_maps" 2>&1 | tail -1
done
for rep in 1 2; do
  for spec in austria:4096 austria:16384 treitlstrasse_v2:65536 columbia:16384 barcelona:65536; do
    echo "== base $spec" | tee -a $OUT/ab.log; RD_SWEEP=$spec python tools/lidar_sweep.py 2>&1 | tail -1 | tee -a $OUT/ab.log
    for v in variants/gpi*.so; do
      echo "== $(basename $v .so) $spec" | tee -a $OUT/ab.log; RD_ENV_LIB=$PWD/$v RD_SWEEP=$spec python tools/lidar_sweep.py 2>&1 | tail -1 | tee -a $OUT/ab.log
    done
  done
done
