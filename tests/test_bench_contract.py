"""CPU: the parts of the bench.py contract that do not need a GPU -- the reference arm's JSON line and the loud failure of the GPU arm without a device.
GPU: --dump-outputs writes the state after exactly W + K steps, the same from run to run, with rho / u updated where the step does not store them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "D3Q19 MLUP/s" and d["unit"] == "MLUP/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] >= 1 and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "block" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "MLUP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["name"] == "urban_fp16s" and d["config"]["lattice"] == [1024, 1024, 256] and d["steps"] == 1 and d["warmup"] == 3  # the B200 arm's config, exactly K and W steps


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
    assert r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_is_the_state_after_the_timed_steps(tmp_path):
    """Two runs with the same arguments dump the same arrays; one more timed step changes them; the dump equals rho / u of the same case stepped
    warmup + steps times through the host API, at the sampled cells."""
    import bench as B
    from latticeurbanwind_b200 import _cabi as A, cases
    from latticeurbanwind_b200.domain import Domain
    name, W = "profile256_fp16s", 3
    dumps = {}
    for run, K in (("a", 4), ("b", 4), ("c", 5)):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", name, "--steps", str(K), "--warmup", str(W), "--also", "", "--sustain", "0",
                            "--no-cpu", "--no-e2e", "--traffic", "off", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == K
        assert sorted(os.listdir(out)) == [f"{name}_rho.npy", f"{name}_u.npy"]
        assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= B.DUMP_BYTES
        dumps[run] = {f: np.load(out / f) for f in os.listdir(out)}
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert all(a[f].dtype == np.float32 and np.array_equal(a[f], b[f]) for f in a)
    assert not np.array_equal(a[f"{name}_u.npy"], c[f"{name}_u.npy"])
    d = B.build_domain(Domain, cases, name, A.ARITH_FAST, 0)
    try:
        d.upload_all(); d.t = 1; d.enqueue_initialize(); d.t = 0
        d.run_steps(W + 5)
        d.download_all()
        cells = B.dump_cells(d.N, 1).astype(np.int64)
        assert np.array_equal(c[f"{name}_rho.npy"], d.rho[cells])
        assert np.array_equal(c[f"{name}_u.npy"], d.u.reshape(3, d.N)[:, cells])
    finally:
        d.close()


@pytest.mark.gpu
def test_dump_outputs_updates_the_fields_a_step_does_not_store(tmp_path, oracle_lib):
    """Without UPDATE_FIELDS (the set of the default workload) the step keeps no rho / u: the dump runs update_fields first and so equals the oracle's
    update_fields after the same steps, bit for bit (STRICT arithmetic), at every cell of a lattice smaller than the sample."""
    import bench as B
    from latticeurbanwind_b200 import _cabi as A, cases
    from latticeurbanwind_b200.domain import CellSet, Domain
    from tests import helpers as H
    O = oracle_lib
    shape, steps, feat = (32, 24, 16), 7, H.FEATURE_SETS["luwnf"]
    assert not feat & B.F_UF and B.dump_cells(int(np.prod(shape)), 1).size == int(np.prod(shape))
    flags, rho, u = H.small_urban(*shape)
    w = cases.relaxation_rate(1e-4)
    ref = H.run_cpu(O.Oracle(), O, shape, A.FP16S, feat, flags, rho, u, steps, w, update_at_end=True)
    assert not np.array_equal(ref[2], u)  # the uploaded fields are not an answer
    with Domain(*shape, precision=A.FP16S, features=feat, w=w, arith=A.ARITH_STRICT, **H.ZONES) as d:
        d.rho[:], d.u[:], d.flags[:] = rho, u, flags
        d.f, d.omega = H.FORCE, H.OMEGA
        d.upload_all(); d.t = 1; d.enqueue_initialize(); d.t = 0
        d.run_steps(steps)
        B.dump_outputs(d, CellSet, A, "small", feat, str(tmp_path), 1)
    assert np.array_equal(np.load(tmp_path / "small_rho.npy"), ref[1])
    assert np.array_equal(np.load(tmp_path / "small_u.npy"), ref[2].reshape(3, -1))
