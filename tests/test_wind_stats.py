"""Pedestrian-level wind statistics (csrc/lbm_wind_stats.cuh, luw_wind_stats_*, luw_column_ground, domain.WindStats, lbm.WindStatistics, LBM_WindStatistics).
CPU: the oracle against an independent float64 restatement and against the C oracle's Welford M2; the kernel source compiled for host threads against the oracle;
the ABI surface. GPU: the device path against the oracle fed with the downloaded samples, against luw_stats, across decompositions and through the C++ host layer.
Bar: bit for bit, except where a float64 restatement is the reference."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from latticeurbanwind_b200 import cases
from oracle import wind_stats_oracle as W
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THRESHOLDS = np.array([0.0, 0.02, 0.04, 0.06, 0.08, 0.1, 0.12, 0.2], np.float32)
HEIGHTS = [0, 2, 5, 30]  # 30 cells runs off the top above the higher roofs of the test lattices


# ---------------------------------------------------------------------------------------------------------------- CPU: oracle
def test_oracle_against_float64_two_pass():
    """Means and co-moments of the float32 oracle == a float64 two-pass computation within float32 tolerance; speed statistics and counts == direct evaluation."""
    samples = H.stats_samples()
    K = H.STATS_N
    orc = W.WindStatsOracle(K, THRESHOLDS)
    for _, u in samples:
        orc.accumulate(u[:K], u[K:2 * K], u[2 * K:])
    X = np.stack([u.reshape(3, K) for _, u in samples]).astype(np.float64)  # [sample, c, k]
    S = len(samples)
    mean = X.mean(0)
    dev = X - mean
    assert np.allclose(orc.mean, mean, rtol=0, atol=2e-8)
    for j, (a, b) in enumerate(W.PAIRS):
        assert np.allclose(orc.C[j], (dev[:, a] * dev[:, b]).sum(0), rtol=0, atol=2e-8), j
    s32 = np.sqrt((X[:, 0].astype(np.float32) ** 2 + X[:, 1].astype(np.float32) ** 2) + X[:, 2].astype(np.float32) ** 2)
    s64 = np.sqrt((X ** 2).sum(1))
    assert np.allclose(orc.mean_s, s64.mean(0), rtol=0, atol=2e-8)
    assert np.allclose(orc.m2_s, ((s64 - s64.mean(0)) ** 2).sum(0), rtol=0, atol=2e-8)
    assert np.array_equal(orc.max_s, s32.max(0))
    for j, t in enumerate(THRESHOLDS):
        assert np.array_equal(orc.exceed[j], (s32 > t).sum(0))
    assert orc.n == S


def test_oracle_diagonal_equals_the_c_oracle_m2(oracle_lib):
    """C_uu / C_vv / C_ww and the means are bit-identical to OracleStats (the restatement of the reference's averaging loop)."""
    K = H.STATS_N
    u_avg, rho_avg, m2u, m2v, m2w = H.stats_run(oracle_lib.OracleStats())
    orc = W.WindStatsOracle(K)
    for _, u in H.stats_samples():
        orc.accumulate(u[:K], u[K:2 * K], u[2 * K:])
    for c, m2 in enumerate((m2u, m2v, m2w)):
        assert np.array_equal(orc.C[c], m2)
        assert np.array_equal(orc.mean[c], u_avg[c::3])


def hand_made_flags():
    """Six columns (Nx = 6, Ny = 1, Nz = 8): ground plane only; a roof at z = 4; an overhang (solid 0, fluid 1-2, solid 3-4); all solid; a TYPE_E side column;
    a roof at z = 6 that a height of 2 cells runs off the top of."""
    Nx, Ny, Nz = 6, 1, 8
    f = np.zeros((Nz, Ny, Nx), np.uint8)
    f[0, 0, :] = 0x01
    f[:5, 0, 1] = 0x01
    f[3:5, 0, 2] = 0x01
    f[:, 0, 3] = 0x01
    f[1:, 0, 4] = 0x02 | 0x04  # TYPE_E (with TYPE_T: only the low two bits classify)
    f[:7, 0, 5] = 0x01
    return f.reshape(-1), (Nx, Ny, Nz)


def test_oracle_column_ground_and_layers_on_hand_made_columns():
    flags, (Nx, Ny, Nz) = hand_made_flags()
    g = W.column_ground(flags, Nx, Ny, Nz)
    assert g[0].tolist() == [1, 5, 1, 0xFFFFFFFF, 1, 7]
    cells, slots = W.layer_cells(flags, Nx, Ny, Nz, g, [0, 1, 2])
    zx = [(int(n) // (Nx * Ny), int(n) % Nx) for n in cells]
    assert zx == [(1, 0), (5, 1), (1, 2), (7, 5), (2, 0), (6, 1), (2, 2), (3, 0), (7, 1)]  # the overhang's z = 3 is solid; TYPE_E and off-top left out
    assert slots.tolist() == [0, 1, 2, 5, 6, 7, 8, 12, 13]
    # owned range of an upper block of a z split: the global z of its first owned layer, and a column solid over the whole block
    assert W.column_ground(flags, Nx, Ny, Nz, z0=1, z1=4, Oz=3)[0].tolist() == [4, 0xFFFFFFFF, 4, 0xFFFFFFFF, 4, 0xFFFFFFFF]


# ---------------------------------------------------------------------------------------------------------------- CPU: kernel source on host threads
EMU_SRC = r'''
#include "cuda_on_host.hpp"
#include "lbm_wind_stats.cuh"
extern "C" {
void emu_column_ground(uint32_t Nx, uint32_t Px, uint32_t Ny, uint32_t z0, uint32_t z1, int32_t Oz, const uint8_t* flags, uint32_t* ground) {
	const unsigned gx = (Nx+255u)/256u;
	emu_blockDim = {256u, 1u, 1u}; emu_gridDim = {gx, Ny, 1u};
	for(unsigned by=0u; by<Ny; by++) for(unsigned bx=0u; bx<gx; bx++) for(unsigned t=0u; t<256u; t++) {
		emu_blockIdx = {bx, by, 0u}; emu_threadIdx = {t, 0u, 0u};
		luw::k_column_ground(Nx, Px, Ny, z0, z1, Oz, flags, ground);
	}
}
void emu_wind_accumulate(uint64_t count, uint64_t N, float inv_n, const float* u, const uint64_t* cell, uint32_t nthr, const float* thr, float* acc, uint32_t* exceed, unsigned grid) {
	luw::WindThresholds t; memset(&t, 0, sizeof(t)); t.count = nthr;
	for(uint32_t j=0u; j<nthr; j++) t.t[j] = thr[j];
	emu_blockDim = {256u, 1u, 1u}; emu_gridDim = {grid, 1u, 1u};
	for(unsigned b=0u; b<grid; b++) for(unsigned i=0u; i<256u; i++) {
		emu_blockIdx = {b, 0u, 0u}; emu_threadIdx = {i, 0u, 0u};
		luw::k_wind_stats_accumulate(count, N, inv_n, u, cell, t, acc, exceed);
	}
}
}
'''


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not os.path.isfile("/usr/local/cuda/include/cuda_fp16.h"):
        pytest.skip("CUDA headers not installed")
    d = tmp_path_factory.mktemp("wind_emu")
    src, so = d / "wind_on_host.cpp", str(d / "libwind_emu.so")
    src.write_text(EMU_SRC)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-w", "-I/usr/local/cuda/include",
                           "-I" + os.path.join(ROOT, "tests", "host_emulation"), "-I" + os.path.join(ROOT, "latticeurbanwind_b200", "csrc"), str(src), "-o", so])
    L = C.CDLL(so)
    L.emu_column_ground.argtypes = [C.c_uint32] * 5 + [C.c_int32, C.c_void_p, C.c_void_p]
    L.emu_wind_accumulate.argtypes = [C.c_uint64, C.c_uint64, C.c_float, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
    return L


def test_kernel_source_column_ground_equals_the_oracle(emu):
    """k_column_ground on a padded-row image (Px = 16 > Nx = 13) of the urban case plus the hand-made columns, whole lattice and an upper z block's owned range."""
    Nx, Ny, Nz, Px = 13, 7, 20, 16
    flags = cases.urban(Nx, Ny, Nz, seed=3, edge=3, pitch=5)[0].reshape(Nz, Ny, Nx).copy()
    hand, _ = hand_made_flags()
    flags[:8, 0, :6] = hand.reshape(8, 1, 6)[:, 0, :]
    flags[:, 3, 4] = 0x01  # an all-solid column
    pitched = np.zeros((Nz, Ny, Px), np.uint8)
    pitched[:, :, :Nx] = flags
    for z0, z1, Oz in ((0, Nz, 0), (1, Nz - 1, 9)):
        got = np.zeros((Ny, Nx), np.uint32)
        emu.emu_column_ground(Nx, Px, Ny, z0, z1, Oz, pitched.ctypes.data, got.ctypes.data)
        assert np.array_equal(got, W.column_ground(flags.reshape(-1), Nx, Ny, Nz, z0, z1, Oz)), (z0, z1, Oz)


def test_kernel_source_accumulate_equals_the_oracle(emu):
    """k_wind_stats_accumulate over seeded samples -- zero velocities and speeds exactly at a threshold included -- == the oracle bit for bit, with a grid-stride
    launch smaller than the list."""
    rng = np.random.default_rng(17)
    N, count = 6000, 1500
    cell = np.sort(rng.choice(N, count, replace=False)).astype(np.uint64)
    acc = np.zeros((12, count), np.float32)
    ex = np.zeros((THRESHOLDS.size, count), np.uint32)
    thr = THRESHOLDS.copy()
    first = None
    orc = None
    for s in range(9):
        u = (np.array([0.05, 0.0, 0.0], np.float32)[:, None] + np.float32(0.04) * rng.standard_normal((3, N)).astype(np.float32)).astype(np.float32)
        u[:, cell[:40]] = 0.0  # zero speed: never above a threshold, not even 0
        if s == 0:
            u[:, cell[40:80]] = np.float32(0.0)
            u[0, cell[40:80]] = np.float32(0.06)  # |u| == 0.06 exactly: not above the 0.06 threshold
            x = u[:, cell]
            first = np.sqrt((x[0] * x[0] + x[1] * x[1]) + x[2] * x[2])
            thr[7] = first[100]  # a threshold that one cell's speed meets exactly
            orc = W.WindStatsOracle(count, thr)
        inv_n = np.float32(1.0) / np.float32(s + 1)
        emu.emu_wind_accumulate(count, N, float(inv_n), u.ctypes.data, cell.ctypes.data, thr.size, thr.ctypes.data, acc.ctypes.data, ex.ctypes.data, 3)
        orc.accumulate(*u[:, cell])
    assert np.array_equal(acc[0:3], orc.mean) and np.array_equal(acc[3:9], orc.C)
    assert np.array_equal(acc[9], orc.mean_s) and np.array_equal(acc[10], orc.m2_s) and np.array_equal(acc[11], orc.max_s)
    assert np.array_equal(ex, orc.exceed)
    assert ex[:, :40].sum() == 0 and acc[11, :40].max() == 0.0


# ---------------------------------------------------------------------------------------------------------------- CPU: ABI surface
def test_abi_symbols_are_bound():
    from latticeurbanwind_b200 import _cabi as A
    L = A.lib()
    out = subprocess.check_output(["nm", "-D", "--defined-only", A.LIB_PATH], text=True)
    for name in ("luw_column_ground", "luw_wind_stats_create", "luw_wind_stats_accumulate", "luw_wind_stats_reset", "luw_wind_stats_download", "luw_wind_stats_destroy"):
        assert f" T {name}\n" in out + "\n" and getattr(L, name).argtypes == A.EXPORTS[name], name


def test_no_device_means_error_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    from latticeurbanwind_b200 import _cabi as A
    L = A.lib()
    g = np.zeros(16, np.uint32)
    assert L.luw_column_ground(None, g.ctypes.data) == A.ERR_NO_DEVICE
    cells, thr = np.zeros(2, np.uint64), np.zeros(1, np.float32)
    h = C.c_void_p()
    assert L.luw_wind_stats_create(None, 2, cells.ctypes.data, 1, thr.ctypes.data, C.byref(h)) == A.ERR_NO_DEVICE and not h.value
    assert L.luw_last_error_string()


# ---------------------------------------------------------------------------------------------------------------- GPU
def _urban(shape, seed=21):
    return cases.urban(*shape, seed=seed, edge=6, pitch=12)


def _domain_run(shape, precision, steps, cells_of, thresholds=THRESHOLDS, stats=False):
    """Urban case on one Domain (STRICT, u stored every step), `steps` steps with a sample after each. cells_of(flags) -> list. Returns (flags, ground,
    cells, WindStats download, per-sample u at the cells, luw_stats download or None)."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, Stats, WindStats
    flags, rho, u = _urban(shape)
    feat = H.FEATURE_SETS["luw"]
    with Domain(*shape, precision=precision, features=feat, w=cases.relaxation_rate(1e-6), arith=A.ARITH_STRICT, **H.ZONES) as d:
        d.rho[:], d.u[:], d.flags[:] = rho, u, flags
        d.f, d.omega = H.FORCE, H.OMEGA
        d.upload_all()
        d.t = 1
        d.enqueue_initialize()
        d.t = 0
        d.read_from_device(A.FIELD_FLAGS)
        d.finish_queue()
        dev_flags = d.flags.copy()
        ground = d.column_ground()
        cells = cells_of(dev_flags, ground)
        ws = WindStats(d, cells, thresholds)
        st = Stats(d) if stats else None
        us = []
        for _ in range(steps):
            d.enqueue_stream_collide()
            d.increment_time_step()
            ws.accumulate()
            if st:
                st.accumulate()
            d.read_from_device(A.FIELD_U)
            d.finish_queue()
            us.append(d.u.reshape(3, -1)[:, cells.astype(np.int64)].copy())
        got = ws.download()
        sgot = st.download() if st else None
        ws.close()
        if st:
            st.close()
        return dev_flags, ground, cells, got, us, sgot


@pytest.mark.gpu
@pytest.mark.parametrize("Nx,precision", [(50, 0), (50, 1), (64, 0), (64, 1)], ids=["padded-fp32", "padded-fp16s", "dense-fp32", "dense-fp16s"])
def test_device_equals_oracle_on_urban_case(Nx, precision):
    shape = (Nx, 40, 48)
    layers = {}

    def cells_of(flags, ground):
        layers["cells"], layers["slots"] = W.layer_cells(flags, *shape, ground, HEIGHTS)
        return layers["cells"]

    flags, ground, cells, got, us, _ = _domain_run(shape, precision, 6, cells_of)
    assert np.array_equal(ground, W.column_ground(flags, *shape))
    assert 0 < cells.size < len(HEIGHTS) * shape[0] * shape[1]
    orc = W.WindStatsOracle(cells.size, THRESHOLDS)
    for u in us:
        orc.accumulate(*u)
    mean_u, com, ms, m2, mx, ex, n = got
    assert n == 6
    assert np.array_equal(mean_u, orc.mean) and np.array_equal(com, orc.C)
    assert np.array_equal(ms, orc.mean_s) and np.array_equal(m2, orc.m2_s) and np.array_equal(mx, orc.max_s) and np.array_equal(ex, orc.exceed)
    assert ex[0].max() == 6 and mx.max() > 0.0  # the wind blows


@pytest.mark.gpu
def test_full_lattice_list_equals_luw_stats():
    """All cells in one list: means and C_uu / C_vv / C_ww identical to luw_stats' mean_u / m2_u on the same run (padded rows)."""
    shape = (50, 24, 20)
    N = int(np.prod(shape))
    _, _, _, got, _, sgot = _domain_run(shape, 1, 5, lambda f, g: np.arange(N, dtype=np.uint64), stats=True)
    mean_u, com = got[0], got[1]
    s_mean, s_m2 = sgot[0].reshape(3, N), sgot[1].reshape(3, N)
    assert np.array_equal(mean_u, s_mean) and np.array_equal(com[:3], s_m2) and got[6] == sgot[3] == 5


def _lbm_wind(shape, D, steps, heights=HEIGHTS, thresholds=THRESHOLDS, features=None):
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import LBM, WindStatistics
    flags, rho, u = _urban(shape)
    lbm = LBM(shape, D=D, precision=A.FP16S, features=H.FEATURE_SETS["luw"] if features is None else features, arith=A.ARITH_STRICT, nu=1e-6, f=H.FORCE,
              omega=H.OMEGA, **H.ZONES)
    lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
    lbm.run(0)
    ws = WindStatistics(lbm, heights, thresholds)
    for _ in range(steps):
        lbm.run(1)
        ws.accumulate()
    out = ws.download()
    out["ground"] = ws.ground
    ws.close()
    lbm.close()
    return out


def _same(a, b):
    for k in a:
        if k == "samples":
            assert a[k] == b[k]
        else:
            assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


@pytest.mark.gpu
@pytest.mark.parametrize("D", [(2, 1, 1), (1, 2, 1), (1, 1, 2)], ids=["2x1x1", "1x2x1", "1x1x2"])
def test_decompositions_equal_the_single_domain(D):
    """In-process decompositions on one device: the same ground, stitched arrays, valid mask and count as the single domain. In [1,1,2] (Nz = 48: blocks of 24
    layers) the ground plane lies in the lower block and the higher roofs (up to z = 45) in the upper one."""
    shape = (64, 40, 48)
    one = _lbm_wind(shape, (1, 1, 1), 5)
    dec = _lbm_wind(shape, D, 5)
    _same(one, dec)
    flags = _urban(shape)[0]
    assert np.array_equal(one["ground"], W.column_ground(flags, *shape))
    valid = np.zeros(one["valid"].size, bool)
    valid[W.layer_cells(flags, *shape, one["ground"], HEIGHTS)[1]] = True
    assert np.array_equal(one["valid"].reshape(-1), valid)
    assert one["samples"] == 5 and one["valid"].any() and not one["valid"].all()
    g = one["ground"]
    assert (g == 1).any() and (g[g != 0xFFFFFFFF] >= 24).any()
    assert np.isnan(one["mean_speed"][~one["valid"]]).all() and (one["exceed"][:, ~one["valid"]] == 0).all()


@pytest.mark.gpu
def test_reset_invalid_arguments_and_stream_order():
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import CellSet, Domain, WindStats, pinned_empty
    shape = (64, 24, 20)
    flags, rho, u = _urban(shape)
    L = A.lib()
    with Domain(*shape, precision=A.FP16S, features=H.FEATURE_SETS["luw"], w=cases.relaxation_rate(1e-6), arith=A.ARITH_STRICT, **H.ZONES) as d:
        d.rho[:], d.u[:], d.flags[:] = rho, u, flags
        d.f, d.omega = H.FORCE, H.OMEGA
        d.upload_all()
        d.t = 1
        d.enqueue_initialize()
        d.t = 0
        cells, _ = W.layer_cells(flags, *shape, W.column_ground(flags, *shape), [0, 3])
        h = C.c_void_p()
        bad_cell, ok_cell = np.array([0, d.N], np.uint64), np.zeros(1, np.uint64)
        nine, nan, neg = np.zeros(9, np.float32), np.array([np.nan], np.float32), np.array([-0.1], np.float32)
        for args in ((2, bad_cell.ctypes.data, 0, None), (1, ok_cell.ctypes.data, 9, nine.ctypes.data), (3, None, 0, None),
                     (1, ok_cell.ctypes.data, 1, nan.ctypes.data), (1, ok_cell.ctypes.data, 1, neg.ctypes.data)):
            assert L.luw_wind_stats_create(d._h, *args, C.byref(h)) == A.ERR_INVALID and not h.value, args
        ws = WindStats(d, cells, THRESHOLDS)
        cs = CellSet(d, cells)
        S = 8
        bufs = [pinned_empty(3 * cells.size, np.float32) for _ in range(S)]
        d.finish_queue()
        n0 = d.launch_count()
        ws.accumulate()
        assert d.launch_count() == n0 + 1
        ws.reset()
        for s in range(S):  # no host synchronisation in the loop: step, sample, gather u of the listed cells (stream-ordered after the sample)
            d.enqueue_stream_collide()
            d.increment_time_step()
            ws.accumulate()
            cs.download(A.FIELD_U, bufs[s])
        d.finish_queue()
        orc = W.WindStatsOracle(cells.size, THRESHOLDS)
        for b in bufs:
            orc.accumulate(*b.reshape(3, -1))
        mean_u, com, ms, m2, mx, ex, n = ws.download()
        assert n == S and np.array_equal(mean_u, orc.mean) and np.array_equal(com, orc.C) and np.array_equal(mx, orc.max_s) and np.array_equal(ex, orc.exceed)
        ws.reset()
        mean_u, com, ms, m2, mx, ex, n = ws.download()
        assert n == 0 and not mean_u.any() and not com.any() and not ms.any() and not m2.any() and not mx.any() and not ex.any()
        cs.close()
        ws.close()


@pytest.mark.gpu
def test_cpp_host_layer_equals_the_python_path(tmp_path):
    """LBM_WindStatistics (C++ host layer, through luw_host_case's LUW_CASE_WIND switch) == lbm.WindStatistics on the same case, single domain and [1,1,2]."""
    from tests.test_cpp_host import build, run_driver
    build()
    shape, steps, samples = (64, 40, 48), 7, 4
    flags, rho, u = _urban(shape)
    feat = H.FEATURE_SETS["core"]
    zones = dict(H.ZONES)
    M, T = len(HEIGHTS) * shape[0] * shape[1], THRESHOLDS.size
    for D in ((1, 1, 1), (1, 1, 2)):
        path = str(tmp_path / "wind.bin")
        env_keep = dict(os.environ)
        os.environ.update(LUW_CASE_WIND=",".join(map(str, HEIGHTS)), LUW_CASE_WIND_THR=",".join(repr(float(t)) for t in THRESHOLDS), LUW_CASE_WIND_OUT=path)
        try:
            run_driver(tmp_path, shape, D, 1, feat, 0, 1e-6, steps, flags, rho, u, zones=zones, stats=samples)
        finally:
            os.environ.clear()
            os.environ.update(env_keep)
        raw = open(path, "rb").read()
        n = np.frombuffer(raw[:8], np.uint64)[0]
        f = np.frombuffer(raw[8:8 + 4 * 12 * M], np.float32)
        o = 8 + 4 * 12 * M
        ex = np.frombuffer(raw[o:o + 4 * T * M], np.uint32)
        valid = np.frombuffer(raw[o + 4 * T * M:o + 4 * T * M + M], np.uint8)
        ground = np.frombuffer(raw[o + 4 * T * M + M:], np.uint32)
        from latticeurbanwind_b200 import _cabi as A
        from latticeurbanwind_b200.lbm import LBM, WindStatistics
        lbm = LBM(shape, D=D, precision=A.FP16S, features=feat, arith=A.ARITH_STRICT, nu=1e-6, f=H.FORCE, omega=H.OMEGA, **zones)
        lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
        lbm.run(0)
        ws = WindStatistics(lbm, HEIGHTS, THRESHOLDS)
        lbm.run(steps - samples)
        for _ in range(samples):
            lbm.run(1)
            ws.accumulate()
        py = ws.download()
        assert np.array_equal(ws.ground.reshape(-1), ground)
        ws.close()
        lbm.close()
        K = (len(HEIGHTS), shape[1], shape[0])
        assert n == py["samples"] == samples
        parts = np.split(f, [3 * M, 9 * M, 10 * M, 11 * M])
        for got, key in zip(parts, ("mean_u", "comoment", "mean_speed", "m2_speed", "max_speed")):
            assert np.array_equal(got.reshape(-1, *K), py[key].reshape(-1, *K), equal_nan=True), (D, key)
        assert np.array_equal(ex.reshape(T, *K), py["exceed"]) and np.array_equal(valid.reshape(K).astype(bool), py["valid"])
