#!/bin/bash
# probe time series: the new GPU tests, smoke(), dev/probes_bench.py (-> profiles/probes_b200.json), bench.py, then the whole GPU suite.
# usage: dev/calls/gpu_probes.sh <output directory>
OUT=${1:?usage: $0 <output directory>}
mkdir -p "$OUT"
timeout 900 python -m pytest tests/test_probes.py -q -m gpu -p no:cacheprovider > "$OUT/pytest_probes_gpu.log" 2>&1; tail -25 "$OUT/pytest_probes_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python dev/probes_bench.py --out "$OUT/probes_b200.json" > /dev/null 2> "$OUT/probes_bench.err"; echo "probes bench rc=$?"; cat "$OUT/probes_b200.json"; tail -c 1500 "$OUT/probes_bench.err"
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench.json"
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > "$OUT/pytest_gpu_all.log" 2>&1; tail -8 "$OUT/pytest_gpu_all.log"
