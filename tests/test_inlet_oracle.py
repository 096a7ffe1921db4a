"""SURVEY 8-f2, oracle level. CPU: oracle/inlet_oracle.py (numpy / Python restatement of the reference's NearestNeighborInterpolator and KNNInterpolatorHD) against
tests/golden/ref_inlet.npz -- velocities returned by the reference's own classes (tests/golden/make_golden_inlet.py). GPU: luw_inlet_nearest / luw_inlet_knn through the
C ABI against the oracle's selections (indices, slot order, max_r2_kept: exact), and the oracle's fit over the KERNEL's selection against the reference's velocities."""
import os

import numpy as np
import pytest

from oracle import inlet_oracle as IO

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_inlet.npz"))
CLOUDS = [0, 1, 2, 3]  # regular grid (ties, coincident samples), jittered, sparse faces, collinear samples (singular fit)
STRIDE = 3  # every third position: the pure-Python selection loop costs ~1 ms per cell and plane sample


def _ulp_close(a, b, ulps=1):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.all((a == b) | (np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)) <= ulps))


@pytest.mark.parametrize("k", CLOUDS)
def test_oracle_reproduces_the_reference_interpolators(k):
    pos = GOLD["pos"][::STRIDE]
    P, U, z = GOLD[f"P_{k}"], GOLD[f"U_{k}"], float(GOLD[f"z_threshold_{k}"][0])
    assert np.array_equal(IO.nearest_eval(P, U, pos, z), GOLD[f"nearest_{k}"][::STRIDE])
    hd = IO.knn_hd_eval(P, U, pos, z)
    want = GOLD[f"hd_{k}"][::STRIDE]
    assert _ulp_close(hd, want), f"{int((hd != want).any(axis=1).sum())} of {len(pos)} velocities differ by more than one unit in the last place"
    assert np.array_equal(hd, want), f"{int((hd != want).any(axis=1).sum())} of {len(pos)} velocities differ in their last bit (a C library whose exp differs from the fixture's)"
    assert np.count_nonzero(want) > len(pos)


@pytest.mark.gpu
@pytest.mark.parametrize("k", CLOUDS)
def test_cuda_searches_equal_the_oracle_and_reproduce_the_reference(k):
    import ctypes as C  # noqa: F401
    from latticeurbanwind_b200 import _cabi as A
    L = A.lib()
    pos = np.ascontiguousarray(GOLD["pos"][::STRIDE])
    P, U, z = GOLD[f"P_{k}"], GOLD[f"U_{k}"], float(GOLD[f"z_threshold_{k}"][0])
    live = np.flatnonzero(pos[:, 2] >= np.float32(z))
    # nearest sample
    cell = np.ascontiguousarray(pos[live].T)
    near = np.zeros(len(live), np.uint32)
    A.check(L.luw_inlet_nearest(0, len(live), cell.ctypes.data, len(P), np.ascontiguousarray(P).ctypes.data, near.ctypes.data))
    got = np.zeros((len(pos), 3), np.float32)
    got[live] = U[near]
    assert np.array_equal(got, GOLD[f"nearest_{k}"][::STRIDE])
    # K = 64: per face plane, the kernel's selection against the oracle's, then the oracle's fit over the kernel's selection against the reference's velocity
    hd = np.zeros((len(pos), 3), np.float32)
    planes = np.array([IO.plane_of(P, pos[c]) for c in live])
    for plane in range(5):
        cells = live[planes == plane]
        if cells.size == 0:
            continue
        idx, q = IO.on_plane(P, plane)
        ab = [(1, 2), (1, 2), (0, 2), (0, 2), (0, 1)][plane]
        cab = np.ascontiguousarray(pos[cells][:, ab].T)
        kept = np.zeros((cells.size, 64), np.uint32); used = np.zeros(cells.size, np.uint32); mr = np.zeros(cells.size, np.float32); ex = np.zeros(cells.size, np.int32)
        A.check(L.luw_inlet_knn(0, cells.size, cab.ctypes.data, len(q), q.ctypes.data, kept.ctypes.data, used.ctypes.data, mr.ctypes.data, ex.ctypes.data))
        for n, c in enumerate(cells):
            exact, okept, omax = IO.knn_select(q, cab[0, n], cab[1, n])
            assert ex[n] == exact, (plane, c)
            if exact >= 0:
                hd[c] = U[idx[exact]]
                continue
            assert used[n] == len(okept) and kept[n, :used[n]].tolist() == okept and mr[n] == omax, (plane, c)
            hd[c] = IO.knn_fit(q, U[idx], kept[n, :used[n]].tolist(), cab[0, n], cab[1, n], mr[n])
    # the oracle's fit over the kernels' selection == the oracle's own evaluation, computed in this process (same exp): bit for bit on any machine
    assert np.array_equal(hd, IO.knn_hd_eval(P, U, pos, z))
    # ... and the reference's velocities from the fixture. The fixture was made with another machine's C library: a weight may differ in its last bit, which a
    # well-conditioned fit does not show in single precision; the collinear cloud (k = 3: singular or nearly singular systems) is left to the CPU test, which
    # runs where the fixture was made, and to baseline/inlet_parity.cpp, which compares with the reference in the same process.
    if k != 3:
        want = GOLD[f"hd_{k}"][::STRIDE]
        assert float(np.abs(hd - want).max()) <= 1e-6, float(np.abs(hd - want).max())


def test_kernel_source_selection_equals_the_oracle_on_adversarial_orders(tmp_path):
    """CPU: csrc/lbm_inlet.cuh compiled for the host (tests/host_emulation) against the oracle's selection loop on sample orders that stress the slot bookkeeping:
    heavy ties (lattice coordinates), samples that approach the cell monotonically (a replacement at every sample), duplicates, a NaN sample; 1 to 500 samples,
    around the K = 64 boundary and the kernel's four-samples-per-trip loop. exact / used / slot order / max_r2_kept must be identical."""
    import ctypes as C
    import subprocess
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emulation")
    if not os.path.isfile("/usr/local/cuda/include/cuda_fp16.h"):
        pytest.skip("CUDA headers not installed")
    so = str(tmp_path / "libinlet_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-w", "-I/usr/local/cuda/include", os.path.join(here, "inlet_on_host.cpp"), "-o", so])
    L = C.CDLL(so)
    L.luw_inlet_knn.argtypes = [C.c_int, C.c_uint64, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5
    rng = np.random.default_rng(5)
    for case in range(40):
        npts, kind = int(rng.choice([1, 3, 63, 64, 65, 66, 67, 130, 257, 500])), case % 5
        if kind == 0:
            q = rng.uniform(-10, 10, (npts, 2))
        elif kind == 1:
            q = rng.integers(-4, 5, (npts, 2)).astype(float)
        elif kind == 2:
            q = np.stack([np.linspace(30, 0.5, npts), np.zeros(npts)], 1)
        elif kind == 3:
            q = np.repeat(rng.uniform(-3, 3, (max(npts // 4, 1), 2)), 4, 0)[:npts]
        else:
            q = rng.uniform(-10, 10, (npts, 2)); q[rng.integers(0, npts)] = [np.nan, 1.0]
        q = np.ascontiguousarray(q, np.float32)
        ncells = 24
        cell = np.ascontiguousarray(rng.integers(-3, 4, (2, ncells)).astype(np.float32) + np.float32(0.0 if kind == 1 else 0.5))
        kept = np.zeros((ncells, 64), np.uint32); used = np.zeros(ncells, np.uint32); mr = np.zeros(ncells, np.float32); ex = np.zeros(ncells, np.int32)
        assert L.luw_inlet_knn(0, ncells, cell.ctypes.data, len(q), q.ctypes.data, kept.ctypes.data, used.ctypes.data, mr.ctypes.data, ex.ctypes.data) == 0
        for c in range(ncells):
            e, k, m = IO.knn_select(q, cell[0, c], cell[1, c])
            assert ex[c] == e, (case, c)
            if e < 0:
                assert used[c] == len(k) and kept[c, :used[c]].tolist() == k and (mr[c] == m or (np.isnan(mr[c]) and np.isnan(m))), (case, kind, c)
