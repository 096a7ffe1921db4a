#!/usr/bin/env python
"""Benchmark of the LBM time step (BASELINE.json metric: D3Q19 MLUP/s at 1/2/4/8 B200 and % of the HBM-bandwidth roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

One "step" = one LBM time step (stream_collide on every cell of the lattice, plus the halo exchange when N > 1).
MLUP/s = cells of the GLOBAL lattice (solids included, halo layers excluded) x steps / seconds / 1e6, the reference's own definition
(FX/info.cpp:66, FX/lbm.cpp:1393).

Workloads (BASELINE.json configs; the per-GPU block is fixed -> weak scaling):
  urban_fp16s        configs[2], the north-star's target step: staggered cube array 1024x1024x256, TYPE_E inflow, bounce-back cubes, Coriolis, nudging,
                     sponge, Smagorinsky LES, FP16S                                                                     (default: the headline line)
  urban_fp16s_uf     the same with UPDATE_FIELDS (rho/u stored every step, +16 B/cell), LUW's shipped semantics
  channel512_fp16s   configs[1]: empty channel 512^3, TYPE_E on the x faces, TYPE_S walls, FP16S DDFs, nu = 1/6 (the upstream README's protocol)
  channel512_fp32 / channel512_fp16c    configs[1] with FP32 / FP16C DDFs
At N = 1 the default run also measures urban_fp16s_uf and the three channel workloads and reports them under `also` (--also '' to skip).
N > 1 (torchrun, one rank per GPU): the lattice is decomposed along z and y first (--decomp for other layouts, see DECOMP); every rank owns
one block of the same local size (halo layers included), halo DDFs move over NVLink.

The JSON line carries, besides the contract keys: `roofline` (dominant kernel, algorithmic bytes per launch / CUDA-event duration against
MEASURED_PEAKS.json), `cpu_baseline` (the reference's kernel text compiled for host threads -- oracle/_ref -- or the C oracle, on a bounded sample),
`e2e` (the same steps driven through the host API one step at a time, each with a pinned-memory upload of that step's inflow boundary field
and a read-back of a probe plane), `clocks`, `gpu_launches`.

--dump-outputs DIR (N = 1): right after the K timed steps of every workload it measures, rho and u (and T on thermal workloads) as the host API returns
them, at a fixed, seeded sample of cells, go to DIR/<workload>_<field>.npy (float32; u is (3, cells)). The inputs are seeded, so two builds run with the
same arguments can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F_UF, F_VF, F_EQ, F_SG, F_NUDGE, F_SPONGE, F_TEMPERATURE = 1, 2, 4, 8, 16, 32, 64
WORKLOADS = {
    # name: (case, local block shape incl. halos, precision, features, oracle feature-set name, nu, description)
    "channel512_fp16s": ("channel", (512, 512, 512), 1, F_EQ, "chan", 1.0 / 6.0, "C2 empty channel 512^3 FP16S (TYPE_E x faces, TYPE_S walls), SRT nu=1/6"),
    "channel512_fp32": ("channel", (512, 512, 512), 0, F_EQ, "chan", 1.0 / 6.0, "C2 empty channel 512^3 FP32 (TYPE_E x faces, TYPE_S walls), SRT nu=1/6"),
    "channel512_fp16c": ("channel", (512, 512, 512), 2, F_EQ, "chan", 1.0 / 6.0, "C2 empty channel 512^3 FP16C (LUW's shipped DDF format), SRT nu=1/6"),
    "urban_fp16s": ("urban", (1024, 1024, 256), 1, F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luwnf", 1e-6,
                    "C3 staggered cube array 1024x1024x256 FP16S, TYPE_E inflow, bounce-back, Coriolis, nudging N=16, sponge N=20, Smagorinsky; rho/u on demand"),
    # BASELINE configs[3] scale: 1.26 G cells per GPU (69 GB of HBM), 10.07 G cells on 8 GPUs; generated and uploaded slab by slab (no host image of the block)
    "city10g_fp16s": ("urban", (1024, 1024, 1200), 1, F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luwnf", 1e-6,
                      "C4 city-sized domain: staggered cube array, 1024x1024x1200 cells per GPU (10.07 G cells on 8 GPUs) FP16S, TYPE_E inflow, bounce-back, Coriolis, nudging, sponge, Smagorinsky"),
    "urban_fp16s_nz": ("urban", (1024, 1024, 256), 1, F_VF | F_EQ | F_SG, "core", 1e-6,
                       "C3 staggered cube array 1024x1024x256 FP16S without the relaxation zones (cost attribution only)"),
    "urban_fp16s_uf": ("urban", (1024, 1024, 256), 1, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luw", 1e-6,
                       "C3 staggered cube array 1024x1024x256 FP16S, full LUW step with UPDATE_FIELDS (+16 B/cell rho/u stores)"),
    # SURVEY 8-f4: the reference's shipped build (TEMPERATURE on). Not a headline workload: one-cell-per-thread kernel, unobserved on a B200 in round 1 (DESIGN.md 4.1)
    "urban_fp16s_thermal": ("urban", (1024, 1024, 256), 1, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE | F_TEMPERATURE, "luwT", 1e-6,
                            "C3 staggered cube array 1024x1024x256 FP16S, full LUW step with UPDATE_FIELDS and thermal D3Q7 transport (TYPE_E cells carry TYPE_T, alpha = 2e-3)"),
    "urban_fp16c_thermal": ("urban", (1024, 1024, 256), 2, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE | F_TEMPERATURE, "luwT", 1e-6,
                            "C3 staggered cube array 1024x1024x256 FP16C + UPDATE_FIELDS + TEMPERATURE: the switches LUW ships (FX/defines.hpp:14-24)"),
    # BASELINE configs[0] size: the example project coarsened to 256 x 256 x 128 (8.4 M cells, 1.3 GB of FP32 DDFs): a launch-latency-sensitive lattice, not a headline
    "profile256_fp32": ("urban", (256, 256, 128), 0, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luw", 1e-6,
                        "C1-sized staggered cube array 256x256x128 FP32, full LUW step with UPDATE_FIELDS (the reference's CPU-runnable configuration)"),
    "profile256_fp16c": ("urban", (256, 256, 128), 2, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luw", 1e-6,
                         "C1-sized staggered cube array 256x256x128 FP16C, full LUW step with UPDATE_FIELDS (the drop-in driver's default precision on an example-sized lattice)"),
    "profile256_fp16s": ("urban", (256, 256, 128), 1, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luw", 1e-6,
                         "C1-sized staggered cube array 256x256x128 FP16S, full LUW step with UPDATE_FIELDS"),
    "urban512_fp32": ("urban", (512, 512, 256), 0, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luw", 1e-6,
                      "staggered cube array 512x512x256 FP32 (10.2 GB of DDFs), full LUW step with UPDATE_FIELDS"),
    "urban_fp16c_uf": ("urban", (1024, 1024, 256), 2, F_UF | F_VF | F_EQ | F_SG | F_NUDGE | F_SPONGE, "luw", 1e-6,
                       "C3 staggered cube array 1024x1024x256 FP16C, full LUW step with UPDATE_FIELDS"),
}
THERMAL_ALPHA = 2.0e-3  # thermal diffusion coefficient of the thermal workload (lattice units); def_w_T = 1/(2 alpha + 1/2), beta = 0 (LUW runs without gravity)
ZONES = dict(downstream_face=2, buffer_N=16, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=20, sponge_inv_tau=0.02)
OMEGA = (0.0, 5.6e-6, 4.7e-6)  # Omega_lbm of SURVEY.md 8d (7.292e-5 * (cos 40, sin 40) * dt)
B_ALG = {0: 153, 1: 77, 2: 77}  # algorithmic bytes per cell-step: 19 DDF loads + 19 stores + 1 flag byte (FX/lbm.cpp:121-122)


def alg_bytes(precision, features):
    """B_ALG, plus 7 g loads + 7 g stores per cell-step with the thermal extension (FX/lbm.cpp:127-128)."""
    return B_ALG[precision] + (14 * (4 if precision == 0 else 2) if features & F_TEMPERATURE else 0)


def thermal_fields(flags, shape):
    """Temperature setup of the thermal workload, in place on a block's flags: every TYPE_E cell also gets TYPE_T (what the case driver does for a WRF deck
    with a T column, FX/setup.cpp:5268-5317); returns T: a stable stratification 1 .. 1.02 over the block height."""
    Nx, Ny, Nz = shape
    flags[(flags & 0x03) == 0x02] |= 0x04
    return np.repeat((np.float32(1.0) + np.float32(0.02) * np.arange(Nz, dtype=np.float32) / np.float32(Nz)).astype(np.float32), Nx * Ny)


def thermal_w_T():
    from latticeurbanwind_b200 import cases
    return float(cases.kernel_literal(np.float32(1.0) / (np.float32(2.0) * np.float32(THERMAL_ALPHA) + np.float32(0.5))))
DTYPE = {0: "f32 arithmetic, f32 DDF storage", 1: "f32 arithmetic, FP16S DDF storage", 2: "f32 arithmetic, FP16C DDF storage"}
# Decomposition per GPU count (the deck's n_gpu). Faces normal to x are the expensive ones in this memory layout (every face cell is a 2-byte element in
# its own 1 KB row: measured 39 + 60 us to extract + insert a 131 k-cell x face against 9 + 9 us for a z face, profiles/), so the defaults split z and y
# first, like a deck author would; --decomp selects any other layout, e.g. the reference README's 2,1,1 / 2,2,1 / 2,2,2.
DECOMP = {"channel": {1: (1, 1, 1), 2: (1, 1, 2), 4: (1, 2, 2), 8: (1, 2, 4)},
          "urban": {1: (1, 1, 1), 2: (1, 2, 1), 4: (1, 4, 1), 8: (1, 8, 1)}}


def kernel_name(tiled, precision, features, arith, cells=0):
    """The step kernel(s) of a workload (csrc/luw_cabi.cu setup_tiles / enqueue_step): FAST FP16 storage runs the lean-loop TMA kernel, and so does the FAST FP32 LES step
    on lattices of 2^25 cells and more; otherwise FP32 and STRICT run the general-loop TMA kernel; thermal domains add k_thermal_g behind the momentum kernel
    (buoyancy-free steps)."""
    if not tiled:
        return "k_stream_collide_thermal" if features & F_TEMPERATURE else "k_stream_collide"
    lean = arith == "fast" and (precision != 0 or (bool(features & F_SG) and not features & F_TEMPERATURE and cells >= 1 << 25))
    k = "k_stream_collide_lean" if lean else "k_stream_collide_tile"
    return k + " + k_thermal_g" if features & F_TEMPERATURE else k


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        try:
            for line in open(self.path):
                c = [v.strip() for v in line.split(",")]
                if len(c) < 8:
                    continue
                try:
                    sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)), reasons=sorted(reasons), samples=len(sm))
        return out


def config_of(workload, arith, D=(1, 1, 1), lattice=None):
    """The `config` object of a JSON line -- the same for the B200 arm and the reference arm of a workload."""
    case, shape, precision, features, fset, nu, desc = WORKLOADS[workload]
    N = shape[0] * shape[1] * shape[2]
    return {"workload": desc, "name": workload, "lattice": list(lattice if lattice is not None else shape), "features": features, "arith": arith, "decomposition": list(D),
            "l2": "state (DDFs %.1f GB per GPU) is far larger than the 126 MB L2; no flush needed" % (19 * N * (4 if precision == 0 else 2) / 1e9)}


# ---------------------------------------------------------------------------------------------------------------- CPU arms
def cpu_engine(precision, fset):
    """The CPU implementation timed beside the GPU: the reference's own kernel text built for host threads if oracle/_ref travelled, else our C port."""
    from oracle import oracle as O
    if O.ref_available(precision, fset):
        return O, O.Reference(precision, fset), "reference"
    return O, O.Oracle(), "port"


def cpu_run(workload, steps, warmup, budget_s=20.0, exact=False):
    """Time `steps` stream_collide calls of the workload's step on a bounded sample: an x-y-complete slab of the same case, Nz cut so that one
    step takes a fraction of a second. `exact`: run exactly `steps` timed and `warmup` untimed steps (the reference arm's contract) and shrink the
    sample instead of the step count until they fit the budget. Returns (MLUP/s, cores, kind, sample description, ms per step, steps)."""
    case, shape, precision, features, fset, nu, _ = WORKLOADS[workload]
    from latticeurbanwind_b200 import cases
    O, eng, kind = cpu_engine(precision, fset)
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    # all host threads, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1 for its workers, which would make this arm 15x slower than it is)
    os.environ["OMP_NUM_THREADS"] = str(cores)
    try:
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)  # the OpenMP runtime may have read the old value already
    except OSError:
        pass
    if hasattr(eng, "set_threads"):
        eng.set_threads(cores)
    Nx, Ny = min(shape[0], 512), min(shape[1], 512)
    Nz = 64 if case == "urban" else 32  # urban: keeps ground, cubes (<= 48 cells high), the nudging shell and the sponge in the sample
    if exact:  # ~2.3 MLUP/s per host thread (measured, g++ build of the kernel text): keep (steps + warmup) steps inside the budget
        while Nx * Ny * Nz * (steps + warmup) / (2.0e6 * cores) > budget_s and Nx > 128:
            Nx, Ny = Nx // 2, Ny // 2
    Ng = (Nx, Ny, Nz)
    flags, rho, u = cases.block_case(case, Ng)
    zones = ZONES if features & (F_NUDGE | F_SPONGE) else {}
    p = O.make_params(Nx, Ny, Nz, precision, features, w=cases.relaxation_rate(nu), **zones)
    fi = np.zeros(19 * p.N, O.ddf_dtype(precision))
    eng.bind(p)
    if features & F_TEMPERATURE:
        gi, T = np.zeros(7 * p.N, O.ddf_dtype(precision)), thermal_fields(flags, Ng)
        eng.set_thermal(thermal_w_T(), 0.0, 1.0)
        eng.initialize_thermal(fi, rho, u, flags, gi, T)
        step = lambda t: eng.stream_collide_thermal(fi, rho, u, flags, t, (0, 0, 0), OMEGA, gi, T)
    else:
        eng.initialize(fi, rho, u, flags)
        step = lambda t: eng.stream_collide(fi, rho, u, flags, t, (0, 0, 0), OMEGA)
    t = 0
    t0 = time.perf_counter()
    step(t); t += 1
    one = time.perf_counter() - t0
    if not exact:
        steps = max(1, min(steps, int(budget_s / max(one, 1e-3))))
        warmup = min(warmup, 2)
    for _ in range(max(0, warmup - 1)):  # the step above was the first warm-up step
        step(t); t += 1
    t0 = time.perf_counter()
    for _ in range(steps):
        step(t); t += 1
    dt = time.perf_counter() - t0
    mlups = p.N * steps / dt / 1e6
    sample = f"{Nx}x{Ny}x{Nz} block of the workload's case ({p.N / 1e6:.1f} M cells), {steps} steps, OpenMP over z-planes on {cores} host threads"
    return mlups, cores, kind, sample, dt / steps * 1e3, steps


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    case, shape, precision, features, fset, nu, desc = WORKLOADS[args.workload]
    mlups, cores, kind, sample, ms, steps = cpu_run(args.workload, args.steps, args.warmup, budget_s=150.0, exact=True)
    D = tuple(int(v) for v in args.decomp.split(",")) if args.decomp else DECOMP[case].get(args.gpus, (1, 1, 1))
    H = tuple(1 if v > 1 else 0 for v in D)
    Ng = tuple((n - 2 * h) * v for n, h, v in zip(shape, H, D))
    line = {"impl": "reference", "metric": "D3Q19 MLUP/s", "value": mlups, "unit": "MLUP/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[precision], "data": "synthetic",
            "config": config_of(args.workload, args.arith, D, Ng),
            "cpu_baseline": {"value": mlups, "unit": "MLUP/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": mlups, "unit": "MLUP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference stream_collide (FX/kernel.cpp text compiled for host threads through oracle/ref_shim) on the box's CPU cores; "
                    "the reference's OpenCL runtime itself needs an OpenCL platform, absent from this image" if kind == "reference" else
                    "CPU restatement of FX/kernel.cpp (oracle/luw_oracle.c) on the box's CPU cores"}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workload", default=os.environ.get("LUW_BENCH_WORKLOAD", "urban_fp16s"), choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--arith", default="fast", choices=["fast", "strict"])
    ap.add_argument("--transport", default="ipc", choices=["ipc", "nccl"], help="N>1: halo payload by remote stores into IPC-mapped peer memory (default) or NCCL send/recv")
    ap.add_argument("--decomp", default="", help="N>1: Dx,Dy,Dz (product = N); default: see DECOMP")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-multi", type=int, default=1, help="N>1: 1 = measure the end-to-end leg on all ranks (per-step boundary upload and probe read-back on every rank), 0 = skip it")
    ap.add_argument("--also", default=None, help="comma-separated extra workloads measured after the headline one (N=1) and reported under `also`; "
                                                 "default: urban_fp16s_uf and the channel workloads when the headline is the default one")
    ap.add_argument("--sustain", type=float, default=2.0, help="seconds of back-to-back steps for the `sustained` figure (0: skip)")
    ap.add_argument("--traffic", default="auto", choices=["auto", "live", "file", "off"],
                    help="roofline.traffic: re-run one step under ncu (live), read the committed capture (file), auto = live when ncu is on PATH")
    ap.add_argument("--traffic-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="N=1: after the timed steps of each workload, write rho / u (/ T) at a fixed, seeded sample of cells to DIR/<workload>_<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs writes what the GPU arm computes on one GPU (--impl b200 --gpus 1)")
    args.warmup = max(args.warmup, 3)
    args.also_default = args.also is None
    if args.also is None:
        args.also = "urban_fp16s_uf,channel512_fp16s,channel512_fp32,channel512_fp16c" if args.workload == "urban_fp16s" and args.gpus == 1 else ""
    if args.impl == "reference":
        return reference_arm(args)
    if args.traffic_child:
        return traffic_child(args)

    from latticeurbanwind_b200 import _cabi as A, cases
    from latticeurbanwind_b200.domain import Domain, CellSet, pinned_empty
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench.py --gpus N ...")
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if A.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the LBM step has no CPU fallback (use --impl reference for the CPU arm)")
    arith = A.ARITH_FAST if args.arith == "fast" else A.ARITH_STRICT
    peak, peak_src = measured_peaks()

    if world == 1:
        res = bench_single(args, args.workload, arith, A, cases, Domain, CellSet, pinned_empty, peak, peak_src, headline=True)
        also = []
        for name in [w for w in args.also.split(",") if w]:
            r = bench_single(args, name, arith, A, cases, Domain, CellSet, pinned_empty, peak, peak_src, headline=False)
            also.append({k: r[k] for k in ("config", "value", "unit", "ms_per_step", "dtype", "roofline", "e2e", "gpu_launches") if k in r})
        if also:
            res["also"] = also
        print(json.dumps(res), flush=True)
        return 0
    return bench_multi(args, arith, A, cases, rank, world, local, peak, peak_src)


def dram_traffic(args, workload):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the step kernel. `live`: this process starts `ncu` on a child copy of
    itself that runs warm-up + one step of the same workload with the same library (so the figure cannot go stale when the kernel changes); `file`: the
    committed capture profiles/traffic_<workload>.json. Returns (bytes or None, where it came from)."""
    import shutil
    mode = args.traffic
    if mode == "off":
        return None, "off"
    ncu = shutil.which("ncu") or ("/usr/local/cuda/bin/ncu" if os.path.isfile("/usr/local/cuda/bin/ncu") else None)
    if mode in ("auto", "live") and ncu:
        cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k", "regex:k_stream_collide", "--launch-skip", "3",
               "--launch-count", "1", "--csv", sys.executable, os.path.abspath(__file__), "--workload", workload, "--arith", args.arith, "--traffic-child"]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
            total, seen = 0.0, 0
            import csv
            for row in csv.reader(r.stdout.splitlines()):
                if len(row) > 3 and any(c.startswith("dram__bytes_") for c in row):
                    name = next(c for c in row if c.startswith("dram__bytes_"))
                    unit, val = row[row.index(name) + 1], float(row[row.index(name) + 2].replace(",", ""))
                    total += val * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}.get(unit, 1.0)
                    seen += 1
            if seen == 2 and total > 0:
                return total, "live: ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum on one launch of this build (child process)"
        except Exception:
            pass
        if mode == "live":
            return None, "live capture failed"
    path = os.path.join(ROOT, "profiles", f"traffic_{workload}.json")
    if os.path.isfile(path):
        try:
            return json.load(open(path))["dram_bytes_per_launch"], f"file: profiles/traffic_{workload}.json (committed ncu capture; may predate the current kernel)"
        except Exception:
            pass
    return None, "unavailable"


def traffic_child(args):
    """Child of dram_traffic(): warm-up + one step of the workload, nothing printed (runs under ncu)."""
    from latticeurbanwind_b200 import _cabi as A, cases
    from latticeurbanwind_b200.domain import Domain, pinned_empty
    arith = A.ARITH_FAST if args.arith == "fast" else A.ARITH_STRICT
    d = build_domain(Domain, cases, args.workload, arith, 0)
    d.upload_all(); d.t = 1; d.enqueue_initialize(); d.t = 0
    d.run_steps(5); d.finish_queue()
    d.close()
    return 0


def build_domain(Domain, cases, workload, arith, device, D=(1, 1, 1), O=(0, 0, 0), Ng=None, pinned=None):
    case, shape, precision, features, fset, nu, desc = WORKLOADS[workload]
    zones = ZONES if features & (F_NUDGE | F_SPONGE) else {}
    d = Domain(*shape, D=D, O=O, precision=precision, features=features, w=cases.relaxation_rate(nu), arith=arith, device=device, **zones)
    if pinned is not None:  # host mirrors in page-locked memory
        d.flags, d.rho, d.u = pinned(d.N, np.uint8), pinned(d.N, np.float32), pinned(3 * d.N, np.float32)
    cases.block_case(case, shape if Ng is None else Ng, O, shape, out=(d.flags, d.rho, d.u))
    d.omega = OMEGA if features & F_VF else (0.0, 0.0, 0.0)
    if features & F_TEMPERATURE:
        if pinned is not None:
            d.T = pinned(d.N, np.float32)
        d.T[:] = thermal_fields(d.flags, shape)
        d.set_thermal(thermal_w_T(), 0.0, 1.0)
    return d


DUMP_BYTES = 64_000_000  # all .npy data of one --dump-outputs run together


def dump_cells(N, workloads):
    """Local cells whose fields --dump-outputs writes: a sorted sample drawn with a fixed seed (every cell of a lattice no larger than the sample), sized
    so that `workloads` dumps of rho + u + T (20 bytes per cell) stay within DUMP_BYTES."""
    count = 1 << 20
    while count * 20 * workloads > DUMP_BYTES and count > 1:
        count //= 2
    if N <= count:
        return np.arange(N, dtype=np.uint64)
    return np.sort(np.random.default_rng(2024).choice(N, count, replace=False)).astype(np.uint64)


def dump_outputs(d, CellSet, A, workload, features, out_dir, workloads):
    """--dump-outputs: what a caller of the host API reads after the steps that ran -- rho / u (/ T), with update_fields first where the step does not
    store them (no UPDATE_FIELDS) -- at the cells of dump_cells(), as float32 DIR/<workload>_<field>.npy; u is (3, cells)."""
    if not features & F_UF:
        d.enqueue_update_fields()
    cs = CellSet(d, dump_cells(d.N, workloads))
    fields = [("rho", A.FIELD_RHO, 1), ("u", A.FIELD_U, 3)] + ([("T", A.FIELD_T, 1)] if features & F_TEMPERATURE else [])
    out = {name: np.empty(comps * cs.count, np.float32) for name, _, comps in fields}
    for name, field, _ in fields:
        cs.download(field, out[name])
    d.finish_queue()
    cs.close()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{workload}_{name}.npy"), a.reshape(3, cs.count) if name == "u" else a)


def bench_single(args, workload, arith, A, cases, Domain, CellSet, pinned_empty, peak, peak_src, headline):
    case, shape, precision, features, fset, nu, desc = WORKLOADS[workload]
    Nx, Ny, Nz = shape
    N = Nx * Ny * Nz
    K, W = args.steps, args.warmup
    d = build_domain(Domain, cases, workload, arith, 0, pinned=pinned_empty)
    try:
        # ---- whole job through the host API: upload of the host images, initialize, K steps, read-back of rho/u (reported as e2e.job)
        t0 = time.perf_counter()
        d.upload_all(); d.t = 1; d.enqueue_initialize(); d.t = 0
        d.finish_queue()
        t_up = time.perf_counter() - t0
        d.run_steps(W); d.finish_queue()
        # ---- value: K steps, state resident in HBM, CUDA events on the domain's stream
        clk = ClockSampler(0); clk.start()
        launches0 = d.launch_count()
        d.timer_begin(); d.run_steps(K); ms = d.timer_end()
        launches = d.launch_count() - launches0
        clocks = clk.stop()
        if args.dump_outputs:
            dump_outputs(d, CellSet, A, workload, features, args.dump_outputs, 1 + len([w for w in args.also.split(",") if w]))
        # ---- roofline pass: the same K steps with an event pair around every main-kernel launch
        d.kernel_timing(True); d.run_steps(K); kms, kn = d.kernel_timing_read(); d.kernel_timing(False)
        mlups = N * K / ms / 1e3
        # the step IS one launch of the step kernel (plus a 4-byte memset node for its strip counter): its average duration over the timed region is ms / K.
        # The second pass brackets every launch with its own event pair; that serialises the launches (no back-to-back overlap of tail and head) and is
        # reported as `kernel_ms_isolated` -- the two must agree to a few per cent.
        kern_ms = ms / K
        achieved = N * alg_bytes(precision, features) / (kern_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": kernel_name(d.uses_tiles(), precision, features, args.arith, N),
                "kernel_ms": kern_ms, "kernel_ms_isolated": kms / max(kn, 1),
                "share_of_step": 1.0,
                "alg_bytes_per_cell": alg_bytes(precision, features), "cells_per_launch": N, "peak_source": peak_src,
                "frac_of_8000_datasheet": achieved / 8000.0}
        # ---- sustained: the driver's K steps are a burst of tens of milliseconds at full boost; the same loop for >= args.sustain seconds shows what power capping leaves
        sustained = None
        if headline and args.sustain > 0:
            n_s = max(K, int(args.sustain * 1e3 / (ms / K)) + 1)
            clk2 = ClockSampler(0); clk2.start()
            d.timer_begin(); d.run_steps(n_s); ms_s = d.timer_end()
            c2 = clk2.stop()
            sustained = {"value": N * n_s / ms_s / 1e3, "unit": "MLUP/s", "steps": n_s, "seconds": ms_s / 1e3, "ms_per_step": ms_s / n_s,
                         "frac": N * alg_bytes(precision, features) / (ms_s / n_s * 1e-3) / 1e9 / peak, "clocks": c2}
        if headline:
            roof["traffic"], roof["traffic_source"] = dram_traffic(args, workload)
        res = {"metric": "D3Q19 MLUP/s", "value": mlups, "unit": "MLUP/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms / K,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[precision], "data": "synthetic",
               "config": config_of(workload, args.arith),
               "roofline": roof, "clocks": clocks, "gpu_launches": int(launches)}
        if sustained:
            res["sustained"] = sustained
        published = {"channel512_fp16s": 55609.0, "channel512_fp32": 42152.0, "channel512_fp16c": 22695.0}.get(workload)
        if published:  # FluidX3D's own B200 number for this protocol (OpenCL; BASELINE.md section 1) -- context, the driver computes its own ratios
            res["config"]["published_reference_b200_mlups"] = published
        # ---- e2e: one host-API call per step, with that step's boundary field going up and a probe plane coming back
        if not args.no_e2e:
            res["e2e"] = e2e_steps(d, CellSet, pinned_empty, A, shape, min(K, 100), t_up, N)
        if headline and not args.no_e2e:
            res["e2e"]["cpp_host"] = cpp_host_e2e(case, shape, precision, features, min(K, 60))
        if headline and not args.no_cpu:
            c_mlups, cores, kind, sample, c_ms, c_steps = cpu_run(workload, 8, 1, budget_s=15.0)
            res["cpu_baseline"] = {"value": c_mlups, "unit": "MLUP/s", "cores": cores, "kind": kind, "sample": sample}
        return res
    finally:
        d.close()


def cpp_host_e2e(case, shape, precision, features, K):
    """The same metric through the reference's C++ API (latticeurbanwind_b200/host: class LBM over the C ABI), driven like FX/setup.cpp drives it: boundary
    conditions through lbm.flags / lbm.u, run(0), then one run(1) per step with a per-step upload of the top boundary plane's velocity from the host mirror and a
    read-back of rho / u on a probe plane into it (host buffers; one synchronisation per step). Separate process: lib/luw_host_bench (host/host_bench.cpp)."""
    exe = os.path.join(ROOT, "latticeurbanwind_b200", "lib", "luw_host_bench")
    if case not in ("urban", "channel") or not os.path.isfile(exe) or features & F_TEMPERATURE:
        return {"unavailable": "luw_host_bench not built or no C++ twin of this case"}
    try:
        r = subprocess.run([exe, case, *map(str, shape), str(precision), str(features), str(K), "5"], capture_output=True, text=True, timeout=600)
        out = json.loads(r.stdout.strip().splitlines()[-1])
        return {"value": out["mlups"], "unit": "MLUP/s", "ms_per_step": out["ms_per_step"], "steps": K, "h2d_bytes_per_step": out["h2d_bytes_per_step"],
                "d2h_bytes_per_step": out["d2h_bytes_per_step"], "probe_mean_ux": out["probe_mean_ux"], "build_and_initialize_s": out["build_and_initialize_s"],
                "api": "LBM::run(1) per step, LBM_Domain::u.enqueue_write_to_device / enqueue_read_from_device(offset, length) (host/lbm.hpp), finish_queue every step",
                "note": "the case is this workload's C++ twin (same lattice, feature set and boundary types; cubes from the same pitch / edge rule)"}
    except Exception as exc:
        return {"unavailable": f"luw_host_bench failed: {exc}"}


def e2e_steps(d, CellSet, pinned_empty, A, shape, K, t_upload_init, N):
    """Every step: H2D of the inflow face's velocity (pinned -> device, scattered into u of the TYPE_E cells of the x=0 face), one time step
    through the same call the host layer makes (luw_stream_collide), D2H of rho/u on the outflow-side probe plane x = Nx-2. Everything is enqueued
    on the domain's stream; the host waits only when a pinned buffer set is reused (the reference's D==1 loop blocks in finish_queue every step,
    FX/lbm.cpp:1288 -- with asynchronous copies that is not needed for correctness)."""
    Nx, Ny, Nz = shape
    yz = (np.arange(Ny, dtype=np.uint64)[None, :] + np.arange(Nz, dtype=np.uint64)[:, None] * np.uint64(Ny)).reshape(-1) * np.uint64(Nx)
    inlet = yz[d.flags[yz.astype(np.int64)] == 2]  # TYPE_E cells of the x = 0 face
    probe = yz + np.uint64(Nx - 2)
    cin, cpr = CellSet(d, inlet), CellSet(d, probe)
    uin = pinned_empty(3 * cin.count, np.float32)
    for c in range(3):
        uin[c * cin.count:(c + 1) * cin.count] = d.u[c * d.N + inlet.astype(np.int64)]
    # a ring of RING pinned buffer sets: step k uploads from / reads back into set k % RING and the host only synchronises when a set comes round again
    # (every RING steps), the way a driver that consumes probe samples asynchronously would; every step still moves its own H2D and D2H bytes
    RING = 4
    uins = [pinned_empty(3 * cin.count, np.float32) for _ in range(RING)]
    for b in uins:
        b[:] = uin
    uprs = [pinned_empty(3 * cpr.count, np.float32) for _ in range(RING)]
    rprs = [pinned_empty(cpr.count, np.float32) for _ in range(RING)]
    upr, rpr = uprs[0], rprs[0]
    # von Karman inlet (on in every default deck): 256 modes on the TYPE_E cells of the x = 0 face, applied before every step like the reference's pre-step update
    # (FX/setup.cpp:538-558, 4897) -- INSIDE the timed loop
    vk, vk_info = None, None
    try:
        from latticeurbanwind_b200.domain import VkInlet
        P, M = int(inlet.size), 256
        rng = np.random.default_rng(5)
        pdv = np.zeros(7 * P, np.float32)
        pdv[0:P] = 0.0; pdv[P:2 * P] = ((inlet // np.uint64(Nx)) % np.uint64(Ny)).astype(np.float32); pdv[2 * P:3 * P] = (inlet // np.uint64(Nx * Ny)).astype(np.float32)
        for c in range(3):
            pdv[(3 + c) * P:(4 + c) * P] = d.u[c * d.N + inlet.astype(np.int64)]
        pdv[6 * P:7 * P] = 0.004
        V = 5 * M
        mdv = np.concatenate([rng.normal(0, 0.3, 3 * V), rng.normal(0, 0.05, V), rng.normal(0, 1.0, 3 * V), rng.uniform(0, 2 * np.pi, 3 * V)]).astype(np.float32)
        vk = VkInlet(d, inlet, np.zeros(P, np.uint8), pdv, mdv, M, V)
        vk.apply(0, 100.0, 101.0, 0.0); d.finish_queue()
        d.timer_begin(); vk.apply(0, 101.0, 102.0, 0.0); vk.apply(0, 102.0, 103.0, 0.0); vk.apply(0, 103.0, 104.0, 0.0); vms = d.timer_end() / 3.0
        vk_info = {"points": P, "modes": M, "apply_ms": vms, "inside_the_timed_loop": True}
    except Exception as exc:  # the loop then runs without it, and says so
        vk, vk_info = None, f"failed: {exc}"
    def step(k):
        r = k % RING
        cin.upload(A.FIELD_U, uins[r])
        if vk is not None:
            vk.apply(0, float(200 + k), float(201 + k), 0.0)
        d.enqueue_stream_collide(); d.increment_time_step()
        cpr.download(A.FIELD_U, uprs[r]); cpr.download(A.FIELD_RHO, rprs[r])
        if r == RING - 1:
            d.finish_queue()
    for k in range(RING):
        step(k)
    t0 = time.perf_counter()
    for k in range(K):
        step(k)
    d.finish_queue()
    dt = time.perf_counter() - t0
    # whole job: upload + initialize (measured above) + K steps + full rho/u read-back
    t1 = time.perf_counter()
    d.read_from_device(A.FIELD_RHO); d.read_from_device(A.FIELD_U); d.finish_queue()
    t_down = time.perf_counter() - t1
    out = {"value": N * K / dt / 1e6, "unit": "MLUP/s", "h2d_bytes_per_step": int(uin.nbytes), "d2h_bytes_per_step": int(upr.nbytes + rpr.nbytes),
           "steps": K, "ms_per_step": dt / K * 1e3, "timer": "host wall clock around K x (boundary upload, von Karman inlet update, step, probe read-back), host sync every 4th step (ring of 4 pinned buffer sets) and at the end",
           "probe_mean_ux": float(upr[:cpr.count].mean()),
           "job": {"upload_init_s": t_upload_init, "h2d_bytes": int(17 * N), "readback_s": t_down, "d2h_bytes": int(16 * N),
                   "note": "one-off per case: full rho/u/flags images up (17 B/cell, pinned), rho/u down (16 B/cell)"}}
    cin.close(); cpr.close()
    if isinstance(vk_info, dict):
        vk_info["share_of_step"] = vk_info["apply_ms"] / (dt / K * 1e3)
    out["job"]["vk_inlet"] = vk_info
    if vk is not None:
        vk.close()
    try:  # one sample of the device-side running statistics (mean / M2 of u, mean of rho: 72 B per cell) next to what it replaces: the read-back above
        from latticeurbanwind_b200.domain import Stats
        st = Stats(d)
        st.accumulate(); d.finish_queue()
        d.timer_begin(); st.accumulate(); st.accumulate(); st.accumulate(); ms = d.timer_end() / 3.0
        out["job"]["stats_sample_ms"] = ms
        out["job"]["stats_sample_gbs"] = 72.0 * N / (ms * 1e-3) / 1e9
        st.close()
    except Exception as exc:  # not part of the metric
        out["job"]["stats_sample_ms"] = f"failed: {exc}"
    return out


def bench_multi(args, arith, A, cases, rank, world, local, peak, peak_src):
    import torch
    import torch.distributed as dist
    from latticeurbanwind_b200.lbm import DistributedLBM
    case, shape, precision, features, fset, nu, desc = WORKLOADS[args.workload]
    torch.cuda.set_device(local)
    # rank 0 prints ONE JSON line on stdout: whatever native libraries write there while the communicators come up (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D0 = tuple(int(v) for v in args.decomp.split(",")) if args.decomp else DECOMP[case][world]
    assert len(D0) == 3 and D0[0] * D0[1] * D0[2] == world, "--decomp must multiply to the number of ranks"
    K, W = args.steps, args.warmup

    def run_decomp(D, with_e2e=False):
        """One weak-scaling measurement: every rank owns a block of the workload's local size (halo layers included) of a lattice decomposed as D."""
        H = tuple(1 if v > 1 else 0 for v in D)
        Ng = tuple((n - 2 * h) * v for n, h, v in zip(shape, H, D))  # global lattice whose blocks have exactly the workload's local size incl. halos
        zones = ZONES if features & (F_NUDGE | F_SPONGE) else {}
        lbm = DistributedLBM(Ng, D, device=local, nu=nu, precision=precision, features=features, arith=arith,
                             omega=OMEGA if features & F_VF else (0.0, 0.0, 0.0), transport=args.transport,
                             **(dict(alpha=THERMAL_ALPHA) if features & F_TEMPERATURE else {}), **zones)
        assert tuple(lbm.Nl) == tuple(shape)
        if int(np.prod(shape)) > 600_000_000:  # C4-sized block: generate and upload 32 planes at a time, the block never exists on the host
            def slabs():
                for z0 in range(0, shape[2], 32):
                    nz = min(32, shape[2] - z0)
                    fl, rh, uu = cases.block_case(case, Ng, (lbm.O[0], lbm.O[1], lbm.O[2] + z0), (shape[0], shape[1], nz))
                    yield z0, fl, rh, uu
            lbm.upload_slabs(slabs())
            dist.barrier()
            lbm.initialize()
            flags_local = None
        else:
            flags, rho, u = cases.block_case(case, Ng, lbm.O, shape)
            T = thermal_fields(flags, shape) if features & F_TEMPERATURE else None  # per-block stratification: a benchmark input, not a physical profile across blocks
            dist.barrier()  # host-side case generation takes seconds and not the same number on every rank: start the first halo exchange together
            lbm.initialize(flags, rho, u, T)
            flags_local = flags
        lbm.run(W)
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        launches0, over0 = lbm.domain.launch_count(), lbm.domain.overlapped_steps()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(lbm._stream); lbm.run(K); e1.record(lbm._stream)  # on the stream the step is enqueued on; it waits for the halo stream's insert at the end of every step
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        dist.barrier(); torch.cuda.synchronize()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        launches, overlapped = lbm.domain.launch_count() - launches0, lbm.domain.overlapped_steps() - over0
        # roofline pass for the step kernel of this rank
        lbm.domain.kernel_timing(True); lbm.run(K); kms, kn = lbm.domain.kernel_timing_read(); lbm.domain.kernel_timing(False)
        kern = torch.tensor([kms / max(kn, 1)], device="cuda")
        dist.all_reduce(kern, op=dist.ReduceOp.MAX)
        e2e = multi_e2e(lbm, flags_local, min(K, 100)) if with_e2e and args.e2e_multi and not args.no_e2e else None
        out = None
        if rank == 0:
            ms, kern_ms = float(ms.item()), float(kern.item())
            Nglob, Nloc = int(np.prod(Ng)), int(np.prod(shape))
            mlups = Nglob * K / ms / 1e3
            achieved = Nloc * alg_bytes(precision, features) / (kern_ms * 1e-3) / 1e9
            halo_bytes = sum(2 * lbm.halo_bytes(A.HALO_FI, a) for a in range(3) if D[a] > 1)
            out = dict(mlups=mlups, ms=ms, kern_ms=kern_ms, achieved=achieved, halo_bytes=int(halo_bytes), launches=int(launches), overlapped=int(overlapped), Ng=Ng, D=D)
            if isinstance(e2e, dict) and "seconds" in e2e:
                e2e = dict(e2e, value=Nglob * e2e["steps"] / e2e.pop("seconds") / 1e6, unit="MLUP/s")
            out["e2e"] = e2e
        lbm.close()
        return out

    def multi_e2e(lbm, flags_local, Ke):
        """The same metric end to end at N ranks: every step, every rank uploads the velocity of its block's inflow-face cells (x = 0 plane, TYPE_E; the x = 1 plane for blocks away from the
        inflow face) from pinned host memory, all ranks step together (halo exchange included), every rank reads rho / u of a probe plane of its block back. Wall clock between two barriers,
        MAX over ranks; the byte counts are sums over the ranks. Everything that can fail (cell sets, pinned buffers, one upload and one read-back) happens BEFORE the ranks
        agree, through an all-reduce, to run the loop -- a rank must not drop out of a collective step loop."""
        ok, why, cin = 1, "", None
        try:
            if flags_local is None:
                raise RuntimeError("the block was uploaded slab by slab and has no host image to take the boundary cells from")
            from latticeurbanwind_b200.domain import CellSet, pinned_empty
            dom = lbm.domain
            Nx, Ny, Nz = shape
            yz = (np.arange(Ny, dtype=np.uint64)[None, :] + np.arange(Nz, dtype=np.uint64)[:, None] * np.uint64(Ny)).reshape(-1) * np.uint64(Nx)
            bc = yz[flags_local[yz.astype(np.int64)] == 2]  # TYPE_E cells of the block's x = 0 plane: the inflow face, as in the N = 1 loop (e2e_steps)
            if bc.size == 0:
                bc = yz + np.uint64(1)  # a block away from the inflow face refreshes its x = 1 plane instead (same bytes, same kernels; the values are the ones already there)
            probe = yz + np.uint64(Nx - 2)
            cin, cpr = CellSet(dom, bc), CellSet(dom, probe)
            RING = 4
            uins = [pinned_empty(3 * cin.count, np.float32) for _ in range(RING)]
            uprs = [pinned_empty(3 * cpr.count, np.float32) for _ in range(RING)]
            rprs = [pinned_empty(cpr.count, np.float32) for _ in range(RING)]
            cin.download(A.FIELD_U, uins[0]); dom.finish_queue()  # the values that are there: the loop re-uploads them (the flow is not disturbed)
            for b in uins[1:]:
                b[:] = uins[0]
            cin.upload(A.FIELD_U, uins[1]); cpr.download(A.FIELD_U, uprs[0]); cpr.download(A.FIELD_RHO, rprs[0]); dom.finish_queue()
        except Exception as exc:
            ok, why = 0, str(exc)
        agree = torch.tensor([ok], device="cuda", dtype=torch.int32)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        if int(agree.item()) != 1:
            return {"unavailable": why or "another rank could not set the loop up"}
        dom = lbm.domain
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(Ke):
            r = k % RING
            cin.upload(A.FIELD_U, uins[r])
            lbm.run(1)
            cpr.download(A.FIELD_U, uprs[r]); cpr.download(A.FIELD_RHO, rprs[r])
            if r == RING - 1:
                dom.finish_queue()
        dom.finish_queue(); torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        nbytes = torch.tensor([uins[0].nbytes, uprs[0].nbytes + rprs[0].nbytes], device="cuda", dtype=torch.int64)
        dist.all_reduce(nbytes, op=dist.ReduceOp.SUM)
        probe_mean = float(uprs[(Ke - 1) % RING][:cpr.count].mean())
        cin.close(); cpr.close()
        return {"seconds": float(dt.item()), "steps": Ke, "h2d_bytes_per_step": int(nbytes[0].item()), "d2h_bytes_per_step": int(nbytes[1].item()), "ms_per_step": float(dt.item()) / Ke * 1e3,
                "probe_mean_ux_rank0": probe_mean,
                "timer": "host wall clock between two barriers around K x (every rank: boundary-cell velocity upload from pinned memory, one step with its halo exchange, probe-plane rho / u read-back), host sync every 4th step, MAX over ranks; bytes summed over ranks"}

    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    r0 = run_decomp(D0, True)
    clocks = clk.stop() if rank == 0 else None
    # the reference README's layouts at 8 GPUs (FX/lbm.cpp:1066-1073: d = x + (y + z*Dy)*Dx), reported beside the default one
    extra = [d for d in ((8, 1, 1), (2, 2, 2)) if world == 8 and not args.decomp and d != D0 and args.also_default]
    also = [run_decomp(d) for d in extra]
    if rank == 0:
        def halo_of(r):
            return {"nvlink_bytes_out_per_gpu_per_step": r["halo_bytes"], "exposed_ms_per_step": r["ms"] / K - r["kern_ms"],
                    "overlapped_with_the_step": r["overlapped"] == K, "note": "y / z exchanges run on a second stream while the interior strips are collided (luw_step_halo_ipc); x faces involve every strip and follow the step"}
        mlups, ms, kern_ms, achieved, Ng, D = r0["mlups"], r0["ms"], r0["kern_ms"], r0["achieved"], r0["Ng"], r0["D"]
        Nloc = int(np.prod(shape))
        res = {"metric": "D3Q19 MLUP/s", "value": mlups, "unit": "MLUP/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[precision], "data": "synthetic",
               "config": dict(config_of(args.workload, args.arith, D, Ng), block_per_gpu_incl_halo=list(shape), halo_transport=args.transport),
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                            "kernel": kernel_name(True, precision, features, args.arith, Nloc), "kernel_ms": kern_ms, "share_of_step": kern_ms / (ms / K), "alg_bytes_per_cell": alg_bytes(precision, features),
                            "cells_per_launch": Nloc, "peak_source": peak_src},
               "halo": halo_of(r0),
               "e2e": r0["e2e"] if isinstance(r0.get("e2e"), dict) and "value" in r0["e2e"] else
                      {"value": mlups, "unit": "MLUP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                       "note": "N>1: the multi-rank loop IS the host-API loop (DistributedLBM.run); the per-step boundary upload / probe read-back leg did not run here: " + str((r0.get("e2e") or {}).get("unavailable", "switched off"))},
               "clocks": clocks, "gpu_launches": r0["launches"]}
        if also:
            res["also"] = [{"decomposition": list(r["D"]), "lattice": list(r["Ng"]), "value": r["mlups"], "unit": "MLUP/s", "ms_per_step": r["ms"] / K, "kernel_ms": r["kern_ms"],
                            "halo": halo_of(r)} for r in also]
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(res), flush=True)
        os.dup2(2, 1)
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
