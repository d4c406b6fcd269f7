#!/bin/bash
# k_lidar work order A/B (RD_LIDAR_ORDER=0 env-major, 1 centre-first) on three batch sizes, then the GPU parity suite
for spec in austria:4096 columbia:16384 treitlstrasse_v2:65536 austria:1024; do
  for rep in 1 2; do for o in 0 1; do
    echo -n "order $o "; RD_LIDAR_ORDER=$o RD_SWEEP=$spec python tools/lidar_sweep.py 2>&1 | tail -1 | cut -c1-150
  done; done
done
timeout 700 python -m pytest tests -x -q -m gpu 2>&1 | tail -3
