"""GPU: cost of the pedestrian-level wind statistics (luw_wind_stats_accumulate) on the C3 urban workload of bench.py (urban_fp16s: 1024 x 1024 x 256 FP16S LES),
for two list sizes:
  layers   4 heights above the local ground or roof x 8 thresholds (the lists lbm.wind_layer_cells builds; about 4 M cells)
  lattice  every cell of the lattice in one list x 8 thresholds (a working set of 48 GB, far above the 126 MB of L2: memory-bound)
Per size: time per accumulate from CUDA events over SAMPLES back-to-back samples after WARMUP, that time as a share of one step measured in the same process,
GB/s against the bytes model below, and that rate as a fraction of a device-to-device copy measured in the same process. Card name and power limit are read
alongside. Prints one JSON line."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload definitions only)
from latticeurbanwind_b200 import _cabi as A, cases  # noqa: E402
from latticeurbanwind_b200.domain import Domain, WindStats  # noqa: E402
from latticeurbanwind_b200.lbm import wind_layer_cells  # noqa: E402

WORKLOAD = "urban_fp16s"
HEIGHTS = [1, 2, 5, 10]  # cells above the ground or roof (2 m cells: 2 - 20 m)
THRESHOLDS = np.linspace(0.01, 0.08, 8).astype(np.float32)  # lattice units
SAMPLES, WARMUP, STEPS = 200, 20, 20


def bytes_per_cell(thresholds):
    """Per listed cell and sample: read u (12 B) and the cell index (8 B); read and write the 12 float accumulators and one counter per threshold."""
    return 12 + 8 + 2 * (4 * 12 + 4 * thresholds)


def copy_peak_gbs():
    """Device-to-device copy of 4 GiB, read + write bytes over event time (median of 5 runs of 5 copies)."""
    import torch
    n = 4 << 30
    src, dst = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    dst.copy_(src)
    rates = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            dst.copy_(src)
        e1.record()
        e1.synchronize()
        rates.append(2 * n * 5 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del src, dst
    torch.cuda.empty_cache()
    return float(np.median(rates))


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    name, power, clock = (v.strip() for v in q.split(","))
    return {"name": name, "power_limit": power, "sm_clock_max": clock}


def timed(d, fn, reps):
    d.timer_begin()
    for _ in range(reps):
        fn()
    return d.timer_end() / reps


def main():
    if A.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    out = {"workload": WORKLOAD, "card": card(), "copy_peak_gbs": copy_peak_gbs(), "samples": SAMPLES, "warmup": WARMUP}
    d = bench.build_domain(Domain, cases, WORKLOAD, A.ARITH_FAST, 0)
    case, shape, precision, features, _, _, desc = bench.WORKLOADS[WORKLOAD]
    out["description"] = desc
    d.upload_all()
    d.t = 1
    d.enqueue_initialize()
    d.t = 0
    d.finish_queue()
    d.run_steps(WARMUP)
    out["step_ms"] = timed(d, lambda: d.run_steps(1), STEPS)
    out["update_fields_ms"] = timed(d, d.enqueue_update_fields, STEPS)  # this workload stores rho / u on demand: a sample needs update_fields first (so does luw_stats)
    ground = d.column_ground()
    layer_cells, _ = wind_layer_cells(d, (0, 0, 0), shape, (1, 1, 1), ground, HEIGHTS)
    for name, cells in (("layers", layer_cells), ("lattice", np.arange(d.N, dtype=np.uint64))):
        ws = WindStats(d, cells, THRESHOLDS)
        timed(d, ws.accumulate, WARMUP)
        ms = timed(d, ws.accumulate, SAMPLES)
        moved = ws.count * bytes_per_cell(THRESHOLDS.size)
        out[name] = {"cells": ws.count, "heights": HEIGHTS if name == "layers" else None, "thresholds": int(THRESHOLDS.size), "accumulate_ms": ms,
                     "share_of_step": ms / out["step_ms"], "bytes_model_per_cell": bytes_per_cell(THRESHOLDS.size), "gbs": moved / (ms * 1e-3) / 1e9,
                     "frac_of_copy_peak": moved / (ms * 1e-3) / 1e9 / out["copy_peak_gbs"], "accumulator_mb": ws.count * (48 + 4 * THRESHOLDS.size) / 2 ** 20}
        if name == "layers":  # (the whole lattice's accumulators would be 21 GB of host arrays)
            _, _, mean_s, _, max_s, _, n = ws.download()
            out[name]["check"] = {"samples": n, "max_speed": float(max_s.max()), "mean_speed_mean": float(mean_s.mean())}
        ws.close()
    d.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
