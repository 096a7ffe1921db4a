"""GPU: cost of Lagrangian tracer particles (luw_particles_advance / _count) on the C3 urban workload of bench.py (urban_fp16s: 1024 x 1024 x 256 FP16S LES,
which does not store rho / u every step, so every advance computes the cell velocities from the DDFs). After SPINUP steps, one street-level emitter box over
the whole ground (z in [1, 4]) releases the particles; releases inside buildings are BURIED, so the ring is sized from a trial release to hold about
10^4, 10^5 and 10^6 ACTIVE particles. Per size, measured with CUDA events in one process:
  advance_ms      one advance (dt = 1, sigma = 0.1), back to back, REPS calls
  count_ms        one count into 8 x 8 x 4-cell bins, back to back, REPS calls
  steps           PAIRS rounds of one step alone and one step followed by an advance, alternating, so clocks and heat affect both alike
Card name and power limit are read alongside (query only). Writes one JSON line to stdout and, with --out, to that file."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "dev"))
import bench  # noqa: E402  (workload definitions only)
from latticeurbanwind_b200 import _cabi as A, cases  # noqa: E402
from latticeurbanwind_b200.domain import Domain, Particles  # noqa: E402
from wall_loads_bench import card, timed  # noqa: E402

WORKLOAD = "urban_fp16s"
SIZES = [10 ** 4, 10 ** 5, 10 ** 6]
SPINUP, REPS, PAIRS = 200, 50, 30
DT, SIGMA, BINS = 1.0, 0.1, (8, 8, 4)


def ground_emitter(shape):
    Nx, Ny, _ = shape
    return np.array([[(Nx - 1) / 2, (Ny - 1) / 2, 2.5, (Nx - 1) / 2, (Ny - 1) / 2, 1.5]])


def measure(d, shape, active_share, size):
    cap = int(np.ceil(size / active_share))
    pt = Particles(d, ground_emitter(shape), cap, 0b011, 0, 7, BINS)
    pt.emit(cap)
    r = {"target_active": size, "capacity": cap, "active": int((pt.state()["state"] == 1).sum())}
    timed(d, lambda: pt.advance(DT, SIGMA), 5)
    r["advance_ms"] = timed(d, lambda: pt.advance(DT, SIGMA), REPS)
    timed(d, pt.count, 5)
    r["count_ms"] = timed(d, pt.count, REPS)
    plain, with_adv = [], []
    for _ in range(PAIRS):  # alternate, in the same call
        plain.append(timed(d, lambda: d.run_steps(1), 1))
        with_adv.append(timed(d, lambda: (d.run_steps(1), pt.advance(DT, SIGMA)), 1))
    base, both = float(np.median(plain)), float(np.median(with_adv))
    r["steps"] = {"plain_ms_median": base, "with_advance_ms_median": both, "advance_overhead_ms": both - base, "advance_overhead_share": both / base - 1.0,
                  "plain_ms_range": [float(min(plain)), float(max(plain))], "with_advance_ms_range": [float(min(with_adv)), float(max(with_adv))]}
    st = pt.state()["state"]
    r["after"] = {name: int((st == k).sum()) for k, name in enumerate(Particles.STATES)}
    pt.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if A.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    out = {"workload": WORKLOAD, "card": card(), "spinup_steps": SPINUP, "reps": REPS, "pairs": PAIRS, "dt": DT, "sigma": SIGMA, "bins": BINS}
    d = bench.build_domain(Domain, cases, WORKLOAD, A.ARITH_FAST, 0)
    _, shape, _, _, _, _, desc = bench.WORKLOADS[WORKLOAD]
    out["description"] = desc
    d.upload_all()
    d.t = 1
    d.enqueue_initialize()
    d.t = 0
    d.finish_queue()
    d.run_steps(SPINUP)
    out["step_ms"] = timed(d, lambda: d.run_steps(1), 20)
    trial = Particles(d, ground_emitter(shape), 1 << 20, 0b011, 0, 7, BINS)
    trial.emit(1 << 20)
    out["active_share_of_release"] = float((trial.state()["state"] == 1).mean())
    trial.close()
    out["sizes"] = {}
    for size in SIZES:
        out["sizes"][str(size)] = measure(d, shape, out["active_share_of_release"], size)
        print(size, json.dumps(out["sizes"][str(size)]), file=sys.stderr, flush=True)
    d.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
