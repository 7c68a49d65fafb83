#!/bin/bash
# Multi-GPU bench on one node under torchrun: bash scripts/gpu_multi.sh N [OUTDIR] (outputs in OUTDIR, default a new temporary directory)
N=${1:-2}
OUT=${2:-$(mktemp -d)}
mkdir -p "$OUT"
nvidia-smi --query-gpu=index,name --format=csv,noheader > "$OUT/multi_gpus_$N.txt"
timeout 1500 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29517 \
  bench.py --gpus $N --steps 20 --warmup 5 > "$OUT/multi_bench_n$N.json" 2> "$OUT/multi_bench_n$N.err"
echo "bench rc=$? (outputs in $OUT)"
cut -c1-300 "$OUT/multi_bench_n$N.json"; tail -3 "$OUT/multi_bench_n$N.err"
python - <<PY
import json
try:
    d = json.load(open("$OUT/multi_bench_n$N.json"))
    print("value", d["value"], "ms/step", d["ms_per_step"], "e2e", d["e2e"]["value"])
    print("work_queue", d.get("work_queue"))
    print("tp", d.get("tensor_parallel"))
except Exception as e:
    print("no json:", e)
PY
if [ "$N" = "2" ]; then timeout 600 python -m pytest tests/test_gpu_tp.py -m gpu -q -x 2>&1 | tail -3; fi
