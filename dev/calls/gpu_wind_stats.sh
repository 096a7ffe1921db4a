#!/bin/bash
# pedestrian-level wind statistics: the new GPU tests, smoke(), dev/wind_stats_bench.py (-> profiles/wind_stats_b200.json), bench.py, then the whole GPU suite.
# usage: dev/calls/gpu_wind_stats.sh <output directory>
OUT=${1:?usage: $0 <output directory>}
mkdir -p "$OUT"
timeout 600 python -m pytest tests/test_wind_stats.py -q -m gpu -p no:cacheprovider > "$OUT/pytest_wind_gpu.log" 2>&1; tail -25 "$OUT/pytest_wind_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python dev/wind_stats_bench.py > "$OUT/wind_stats_bench.json" 2> "$OUT/wind_stats_bench.err"; echo "wind bench rc=$?"; cat "$OUT/wind_stats_bench.json"; tail -c 1500 "$OUT/wind_stats_bench.err"
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench.json"
timeout 1200 python -m pytest tests -q -m gpu -p no:cacheprovider > "$OUT/pytest_gpu_all.log" 2>&1; tail -8 "$OUT/pytest_gpu_all.log"
