#!/usr/bin/env bash
# A/B of two builds of libdsoft.so on ONE board (gpurun -- bash scripts/ab_lib.sh <variant name> [tag]): the GPU test
# suite on the in-tree build, then the bench line of each build, alternating twice.
set -x
var=${1:-variant}
tag=${2:-ab}
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -q -x 2>&1 | tail -6 > gpurun_out/${tag}_gpu_tests.log; cat gpurun_out/${tag}_gpu_tests.log
for r in 1 2; do
  timeout 300 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/${tag}_new_$r.json 2> gpurun_out/${tag}_new_$r.err
  DSOFT_LIB=$PWD/gpurun_variants/libdsoft_${var}.so timeout 300 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/${tag}_${var}_$r.json 2> gpurun_out/${tag}_${var}_$r.err
done
for f in new_1 ${var}_1 new_2 ${var}_2; do python -c "
import json; d=json.loads(open('gpurun_out/${tag}_$f.json').read().strip().splitlines()[-1]); print('$f', round(d['ms_per_step'],3), {k: v['ms'] for k, v in d['kernels'].items()}, d['clocks']['sm_mhz'], d['clocks'].get('power_w'))"; done
