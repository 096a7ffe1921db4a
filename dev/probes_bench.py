"""GPU: cost of probe time series (luw_probes_sample / _drain) on the C3 urban workload of bench.py (urban_fp16s: 1024 x 1024 x 256 FP16S LES, which does not
store rho / u every step), against the route a case driver has without it: update_fields over the lattice, a cell-set gather of rho and u, a synchronous
download. Probe sets: P = 64, 4 096 and 262 144 seeded random cells, and the cells of the pedestrian-level layers of dev/wind_stats_bench.py (4 heights above
the local ground or roof, about 4.2 M cells). Per set, measured with CUDA events / a host clock around synchronised work in one process:
  sample_ms       the sample call alone, back to back (ring drained outside the timed span)
  steps           PAIRS rounds of one step alone and one step followed by a sample, alternating, so clocks and heat affect both alike
  drain_ms        host time of luw_probes_drain of a full ring (synchronous device-to-host copy), median of DRAINS
  route           the same alternating pairs with update_fields + cell-set download of rho and u + synchronisation after the step instead of a sample
The byte model per probe and sample is 2 x 19 B of DDFs read (pairs of FP16 DDFs at two cells), 16 B written and an 8 B index: the large-P rate is
reported against it and against a device-to-device copy measured in the same process. Card name and power limit are read alongside (query only).
Writes one JSON line to stdout and, with --out, to that file."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "dev"))
import bench  # noqa: E402  (workload definitions only)
from latticeurbanwind_b200 import _cabi as A, cases  # noqa: E402
from latticeurbanwind_b200.domain import CellSet, Domain, Probes  # noqa: E402
from latticeurbanwind_b200.lbm import wind_layer_cells  # noqa: E402
from wall_loads_bench import card, copy_peak_gbs, timed  # noqa: E402

WORKLOAD = "urban_fp16s"
SIZES = [64, 4096, 262144]
HEIGHTS = [1, 2, 5, 10]  # the layers of dev/wind_stats_bench.py
REPS, WARMUP, PAIRS, DRAINS = 100, 10, 30, 5
RING_BYTES = 512 << 20  # ring capacity per set: at most 512 MB, at most 256 samples
BYTES_PER_PROBE = 2 * 19 + 16 + 8


def measure(d, cells, step_ms):
    P = int(cells.size)
    cap = int(max(1, min(256, RING_BYTES // (16 * P))))
    pr = Probes(d, cells, cap)
    r = {"probes": P, "capacity": cap}
    pending = [0]

    def sample():
        if pending[0] == cap:
            pr.drain()
            pending[0] = 0
        pr.sample()
        pending[0] += 1

    timed(d, sample, WARMUP)
    reps, rounds = min(REPS, cap), max(1, REPS // min(REPS, cap))
    per = []
    for _ in range(min(rounds, 10)):
        pr.drain()
        pending[0] = 0
        per.append(timed(d, sample, reps))
    r["sample_ms"] = float(np.median(per))
    r["sample_reps"] = [reps, len(per)]
    r["sample_share_of_step"] = r["sample_ms"] / step_ms
    r["gbs_model"] = P * BYTES_PER_PROBE / (r["sample_ms"] * 1e-3) / 1e9
    drains = []
    for _ in range(DRAINS):
        pr.drain()
        for _ in range(cap):
            pr.sample()
        d.finish_queue()
        t0 = time.perf_counter()
        pr.drain()
        drains.append((time.perf_counter() - t0) * 1e3)
    pending[0] = 0
    r["drain_full_ring_ms"] = float(np.median(drains))
    r["drain_mb"] = cap * 16 * P / 2 ** 20
    cs = CellSet(d, cells)
    rho, u = np.empty(P, np.float32), np.empty(3 * P, np.float32)

    def route():  # what a case driver does without probes
        d.enqueue_update_fields()
        cs.download(A.FIELD_RHO, rho)
        cs.download(A.FIELD_U, u)
        d.finish_queue()

    route()
    plain, with_probe, plain_host, with_route = [], [], [], []
    for _ in range(PAIRS):  # alternate, in the same call
        plain.append(timed(d, lambda: d.run_steps(1), 1))
        if pending[0] == cap:  # drains stay out of the timed spans
            pr.drain()
            pending[0] = 0
        with_probe.append(timed(d, lambda: (d.run_steps(1), sample()), 1))
        t0 = time.perf_counter()
        d.run_steps(1)
        d.finish_queue()
        plain_host.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        d.run_steps(1)
        route()
        with_route.append((time.perf_counter() - t0) * 1e3)
    base = float(np.median(plain))
    r["steps"] = {"plain_ms_median": base, "with_sample_ms_median": float(np.median(with_probe)),
                  "sample_overhead_ms": float(np.median(with_probe)) - base, "sample_overhead_share": float(np.median(with_probe)) / base - 1.0}
    hbase = float(np.median(plain_host))
    r["route"] = {"plain_host_ms_median": hbase, "step_plus_route_ms_median": float(np.median(with_route)), "route_overhead_ms": float(np.median(with_route)) - hbase,
                  "route_overhead_share": float(np.median(with_route)) / hbase - 1.0,
                  "note": "host clock around step + synchronise, against step + update_fields + gather + synchronous download"}
    pr.drain()
    # the first sample equals update_fields + gather (the bit-identity the tests check, here at the benchmark's size)
    pr.sample()
    got = pr.drain()[0]
    route()
    r["equals_update_fields"] = bool(np.array_equal(got[0].view(np.uint32), rho.view(np.uint32)) and np.array_equal(got[1:].reshape(-1).view(np.uint32), u.view(np.uint32)))
    cs.close()
    pr.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if A.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    out = {"workload": WORKLOAD, "card": card(), "copy_peak_gbs": copy_peak_gbs(), "reps": REPS, "pairs": PAIRS, "bytes_model_per_probe": BYTES_PER_PROBE}
    d = bench.build_domain(Domain, cases, WORKLOAD, A.ARITH_FAST, 0)
    _, shape, precision, features, _, _, desc = bench.WORKLOADS[WORKLOAD]
    out["description"] = desc
    d.upload_all()
    d.t = 1
    d.enqueue_initialize()
    d.t = 0
    d.finish_queue()
    d.run_steps(WARMUP)
    out["step_ms"] = timed(d, lambda: d.run_steps(1), 20)
    out["update_fields_ms"] = timed(d, d.enqueue_update_fields, 20)
    rng = np.random.default_rng(2026)
    sets = [(f"P{P}", np.sort(rng.integers(0, d.N, P)).astype(np.uint64)) for P in SIZES]
    layer_cells, _ = wind_layer_cells(d, (0, 0, 0), shape, (1, 1, 1), d.column_ground(), HEIGHTS)
    sets.append(("layers", layer_cells))
    out["sets"] = {}
    for name, cells in sets:
        out["sets"][name] = measure(d, cells, out["step_ms"])
        out["sets"][name]["frac_of_copy_peak"] = out["sets"][name]["gbs_model"] / out["copy_peak_gbs"]
        print(name, json.dumps(out["sets"][name]), file=sys.stderr, flush=True)
    d.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
