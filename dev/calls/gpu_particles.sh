#!/bin/bash
# tracer particles: the new GPU tests, smoke(), dev/particles_bench.py (-> profiles/particles_b200.json), bench.py against the parent commit (built in
# $PARENT, alternating), then the whole GPU suite. Stages can be skipped: STAGES="tests bench" runs only those.
# usage: dev/calls/gpu_particles.sh <output directory> [parent tree]
OUT=${1:?usage: $0 <output directory> [parent tree]}
PARENT=${2:-}
STAGES=${STAGES:-"tests smoke bench parent all"}
mkdir -p "$OUT"
has() { [[ " $STAGES " == *" $1 "* ]]; }
if has tests; then timeout 1200 python -m pytest tests/test_particles.py -q -m gpu -p no:cacheprovider -s > "$OUT/particles_pytest_gpu.log" 2>&1; tail -30 "$OUT/particles_pytest_gpu.log"; fi
if has smoke; then timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2; fi
if has bench; then timeout 900 python dev/particles_bench.py --out "$OUT/particles_b200.json" > /dev/null 2> "$OUT/particles_bench.err"; echo "particles bench rc=$?"; cat "$OUT/particles_b200.json"; tail -c 1500 "$OUT/particles_bench.err"; fi
if has parent && [ -n "$PARENT" ]; then
  for k in 1 2; do
    timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_new_$k.json" 2> "$OUT/bench_new_$k.err"; echo "new run $k rc=$?: $(python -c "import json,sys; print(json.loads(open(sys.argv[1]).read().splitlines()[-1])['value'])" "$OUT/bench_new_$k.json")"
    (cd "$PARENT" && timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5) > "$OUT/bench_parent_$k.json" 2> "$OUT/bench_parent_$k.err"; echo "parent run $k rc=$?: $(python -c "import json,sys; print(json.loads(open(sys.argv[1]).read().splitlines()[-1])['value'])" "$OUT/bench_parent_$k.json")"
  done
  nvidia-smi -i 0 --query-gpu=name,power.limit --format=csv,noheader
fi
if has all; then timeout 2400 python -m pytest tests -q -m gpu -p no:cacheprovider > "$OUT/pytest_gpu_all.log" 2>&1; tail -8 "$OUT/pytest_gpu_all.log"; fi
