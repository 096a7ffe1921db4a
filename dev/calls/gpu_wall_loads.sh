#!/bin/bash
# wind loads on buildings: the new GPU tests, smoke(), dev/wall_loads_bench.py (-> profiles/wall_loads_b200.json), bench.py, then the whole GPU suite.
# usage: dev/calls/gpu_wall_loads.sh <output directory>
OUT=${1:?usage: $0 <output directory>}
mkdir -p "$OUT"
timeout 900 python -m pytest tests/test_wall_loads.py -q -m gpu -p no:cacheprovider > "$OUT/pytest_wall_gpu.log" 2>&1; tail -25 "$OUT/pytest_wall_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python dev/wall_loads_bench.py --out "$OUT/wall_loads_b200.json" > /dev/null 2> "$OUT/wall_loads_bench.err"; echo "wall bench rc=$?"; cat "$OUT/wall_loads_b200.json"; tail -c 1500 "$OUT/wall_loads_bench.err"
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench.json"
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > "$OUT/pytest_gpu_all.log" 2>&1; tail -8 "$OUT/pytest_gpu_all.log"
