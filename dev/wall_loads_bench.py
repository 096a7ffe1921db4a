"""GPU: cost of the wind loads on buildings (luw_solid_surface, luw_wall_loads_accumulate) on the C3 urban workload of bench.py (urban_fp16s: 1024 x 1024 x 256
FP16S LES), labels as lbm.WallLoads builds them (576 footprints + terrain). Measured with CUDA events in one process:
  surface       the surface enumeration (both calls of luw_solid_surface), once
  accumulate    the accumulate call alone, SAMPLES back to back after WARMUP (ring drained outside the timed span)
  steps         PAIRS rounds of one step without and one step with an accumulate after it, alternating, so clocks and heat affect both alike
  kernels       device time per launch of each wall-load kernel, from torch.profiler in a separate pass
The per-sample rate is reported against the byte model below and as a fraction of a device-to-device copy measured in the same process; card name and
power limit are read alongside (query only). Writes one JSON line to stdout and, with --out, to that file."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload definitions only)
from latticeurbanwind_b200 import _cabi as A, cases  # noqa: E402
from latticeurbanwind_b200.domain import Domain, WallLoads  # noqa: E402
from latticeurbanwind_b200.lbm import footprint_labels, footprint_ref_points  # noqa: E402

WORKLOAD = "urban_fp16s"
SAMPLES, WARMUP, STEPS, PAIRS = 200, 20, 20, 50


def bytes_per_cell(ddf_bytes):
    """Per listed cell and sample, HBM: cell index (8) + link mask (4) + 19 DDFs + F written (12) + mean / M2 read and written (2 x 24) in the per-cell kernel;
    cell index (8) + F (12) read again by the chunk sums. The chunk and label partials (48 B per 32 cells) are left out."""
    return 8 + 4 + 19 * ddf_bytes + 12 + 48 + 8 + 12


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


def kernel_ms(d, fn, reps):
    """Mean device time per launch of every wall-load kernel over `reps` calls of fn, from torch.profiler (CUDA activities), in a pass of its own."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    d.finish_queue()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        d.finish_queue()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if "k_wall" in e.name and e.time_range.elapsed_us() > 0), key=lambda e: e.time_range.start)
    out, segment = {}, 0
    for e in ev:
        name = e.name.split("(")[0].split("::")[-1].replace("void ", "")
        if name.startswith("k_wall_segments"):  # launched twice per sample: the groups, then the labels
            name += " (groups)" if segment % 2 == 0 else " (labels)"
            segment += 1
        r = out.setdefault(name, {"ms": 0.0, "launches": 0})
        r["ms"] += e.time_range.elapsed_us() / 1e3
        r["launches"] += 1
    for r in out.values():
        r["ms"] /= r["launches"]
    return out


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
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if A.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    out = {"workload": WORKLOAD, "card": card(), "copy_peak_gbs": copy_peak_gbs(), "samples": SAMPLES, "warmup": WARMUP, "pairs": PAIRS}
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
    out["update_fields_ms"] = timed(d, d.enqueue_update_fields, STEPS)  # what a sample would cost first if it needed rho / u (it does not)
    d.solid_surface(0)  # first call: module load and allocations out of the timed span
    d.timer_begin()
    cells = d.solid_surface(0)
    out["surface_ms"] = d.timer_end()
    c = cells.astype(np.int64)
    x, y, z = c % d.Nx, (c // d.Nx) % d.Ny, c // (d.Nx * d.Ny)
    ground = d.column_ground()
    col = footprint_labels(ground, 0)
    L = int(col.max()) + 1
    labels = np.where(z > 0, col[y, x], 0).astype(np.uint32)
    order = np.lexsort((cells, labels))
    wl = WallLoads(d, cells[order], labels[order], L, footprint_ref_points(col, L, 0), 0, SAMPLES + WARMUP)
    out["surface"] = {"cells": int(cells.size), "ground_cells": int((z == 0).sum()), "building_cells": int((labels != 0).sum()), "labels": L}
    timed(d, wl.accumulate, WARMUP)
    wl.drain()
    ms = timed(d, wl.accumulate, SAMPLES)
    series = wl.drain()
    ddf_bytes = 4 if precision == A.FP32 else 2
    moved = cells.size * bytes_per_cell(ddf_bytes)
    out["accumulate"] = {"ms": ms, "share_of_step": ms / out["step_ms"], "bytes_model_per_cell": bytes_per_cell(ddf_bytes), "gbs": moved / (ms * 1e-3) / 1e9,
                         "frac_of_copy_peak": moved / (ms * 1e-3) / 1e9 / out["copy_peak_gbs"],
                         "check": {"drained": int(series.shape[0]), "building_Fx_sum_last": float(series[-1, 1:, 0].sum()), "terrain_Fx_last": float(series[-1, 0, 0])}}
    try:  # per kernel, in a pass of its own (the profiler is off for every other number)
        out["accumulate"]["kernels"] = kernel_ms(d, wl.accumulate, 20)
    except Exception as e:  # noqa: BLE001  (the breakdown is supplementary; the event timings above stand without it)
        out["accumulate"]["kernels"] = {"error": repr(e)}
    wl.drain()
    wl.reset()
    plain, with_acc = [], []
    for _ in range(PAIRS):  # alternate, in the same call
        plain.append(timed(d, lambda: d.run_steps(1), 1))
        with_acc.append(timed(d, lambda: (d.run_steps(1), wl.accumulate()), 1))
        if len(with_acc) % (SAMPLES + WARMUP) == 0:
            wl.drain()
    out["steps"] = {"plain_ms_median": float(np.median(plain)), "with_accumulate_ms_median": float(np.median(with_acc)),
                    "overhead_ms": float(np.median(with_acc) - np.median(plain)), "overhead_share": float(np.median(with_acc) / np.median(plain) - 1.0)}
    wl.close()
    d.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
