#!/usr/bin/env bash
# A/B of the shared symmetric tiles on one node of N GPUs (bash scripts/symw_ab.sh N tag):
# NCCL parity tests, then the bench line with the exchanges next to the CLIP kernels and with DSOFT_SYM_W=0.
set -x
n=${1:-2}
tag=${2:-r04}
mkdir -p gpurun_out
run() { timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port $((29500 + RANDOM % 400)) "$@"; }
if [ "$n" = 8 ]; then k="-k eight_gpu"; else k=""; fi
timeout 400 python -m pytest tests/test_gpu_dist.py tests/test_gpu_symw.py -m gpu -q $k 2>&1 | tail -5 > gpurun_out/${tag}_dist${n}_tests.log; cat gpurun_out/${tag}_dist${n}_tests.log
run bench.py --gpus $n --steps 20 --warmup 5 --no-cpu-baseline > gpurun_out/${tag}_bench_n${n}.json 2> gpurun_out/${tag}_n${n}.err
DSOFT_SYM_W=0 run bench.py --gpus $n --steps 20 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/${tag}_bench_n${n}_nosymw.json 2> gpurun_out/${tag}_n${n}_nosymw.err
for f in bench_n${n} bench_n${n}_nosymw; do python -c "
import json; d=json.loads(open('gpurun_out/${tag}_$f.json').read().strip().splitlines()[-1]); print('$f', d['ms_per_step'], d['value'], (d.get('e2e') or {}).get('value'), d['step_roofline']['serial_ms_per_step'], d['step_roofline']['tile_kernel_ms_per_serial_step'], d['clocks'])"; tail -3 gpurun_out/${tag}_n${n}*.err | cut -c1-300; done
