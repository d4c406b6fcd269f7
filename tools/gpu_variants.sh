#!/bin/bash
# A/B timing of prebuilt library variants (variants/*.so) + source-level ncu of the occupancy kernel
OUT=gpurun_out/${1:-var}; mkdir -p $OUT
for v in variants/*.so; do
  for rep in 1 2; do
    echo "== $v" | tee -a $OUT/variants.log
    RD_ENV_LIB=$PWD/$v RD_SWEEP=austria:4096 python tools/lidar_sweep.py 2>&1 | tail -1 | tee -a $OUT/variants.log
  done
done
timeout 600 python -m pytest tests -x -q -m gpu 2>&1 | tail -3
timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_occupancy -s 2 -c 1 -o $OUT/prof_occ -f \
   python bench.py --obs lidar_occupancy --envs 4096 --steps 4 --warmup 3 --no-cpu-baseline --e2e-steps 2 > $OUT/ncu_occ.log 2>&1; echo "ncu rc=$?"
timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_step -s 5 -c 1 -o $OUT/prof_step -f \
   python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-steps 2 > $OUT/ncu_step.log 2>&1; echo "ncu rc=$?"
python bench.py --no-cpu-baseline 2>/dev/null | python -c "import json,sys; d=json.loads(sys.stdin.read()); print(d['value'], d['kernel_ms'], d['e2e']['value'])"
