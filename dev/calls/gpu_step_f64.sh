#!/bin/bash
# one-step FAST / STRICT parity against the float64 reference: the new GPU tests (-> parity_measured.jsonl), smoke(), bench.py, then the whole GPU suite.
# usage: dev/calls/gpu_step_f64.sh <output directory>
OUT=${1:?usage: $0 <output directory>}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
timeout 900 python -m pytest tests/test_step_f64.py -q -m gpu -p no:cacheprovider -rf > "$OUT/pytest_step_f64_gpu.log" 2>&1; tail -4 "$OUT/pytest_step_f64_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench.json"
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > "$OUT/pytest_gpu_all.log" 2>&1; tail -8 "$OUT/pytest_gpu_all.log"
