#!/usr/bin/env bash
# Diagnostic (gpurun --gpus 2 -- bash scripts/diag_runahead.sh): headline loop vs host enqueue time vs the same loop
# repeated after the per-kernel pass, for the two phase schedules of a DSOFT_SYM_W plan.
n=${1:-2}
mkdir -p gpurun_out
run() { timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port $((29500 + RANDOM % 400)) "$@"; }
for arm in "X=1" "DSOFT_CONCURRENCY=1"; do
  echo "== $arm"
  env $arm DSOFT_BENCH_REPEAT=1 bash -c "$(declare -f run); n=$n; run bench.py --gpus $n --steps 20 --warmup 5 --no-cpu-baseline --no-e2e" 2>&1 >/dev/null | grep "\[bench\]"
done
