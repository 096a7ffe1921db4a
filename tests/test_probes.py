"""Probe time series (csrc/lbm_probes.cuh, luw_probes_*, domain.Probes, lbm.Probes, lbm.probe_columns, LBM_Probes).
CPU: the kernel source compiled for host threads against the C oracle's update_fields at listed cells; the ABI surface; point ownership over decompositions;
probe_columns. GPU: a sample against luw_update_fields + a cell-set download on the same domain, no side effect on the fields, the C oracle, stream order,
ring and argument errors, decompositions, and the C++ host layer. Bar: bit for bit everywhere."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from latticeurbanwind_b200 import cases
from latticeurbanwind_b200.lbm import _local_index, probe_columns, probe_owners, split

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UF, VF, EQ, SG, ZONE_BITS, TEMPERATURE = 1, 2, 4, 8, 16 | 32, 64
FEATS = [0, 4, 5, 14, 15]


def _features(feat, thermal=False):
    """The feature sets under test, with nudging and the top sponge on wherever the volume force is (update_fields must ignore them)."""
    return feat | (ZONE_BITS if feat & VF else 0) | (TEMPERATURE if thermal else 0)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------------------------- CPU: kernel source on host threads
EMU_SRC = r'''
#include "kernels_on_host.cpp"
#include "lbm_probes.cuh"
template<int P, uint32_t F, bool TH> static void run_probe(const DomainConst& c, const StepArgs& a, uint64_t count, const uint64_t* cell, float* out, unsigned grid) {
	emu_blockDim = {256u, 1u, 1u}; emu_gridDim = {grid, 1u, 1u};
	for(unsigned b=0u; b<grid; b++) for(unsigned i=0u; i<256u; i++) { emu_blockIdx = {b, 0u, 0u}; emu_threadIdx = {i, 0u, 0u}; k_probe_sample<P, F, TH>(c, a, count, cell, out); }
}
template<int P, bool TH> static void pick(const DomainConst& c, const StepArgs& a, uint64_t count, const uint64_t* cell, float* out, unsigned grid) {
	if(c.features&F_UPDATE_FIELDS) run_probe<P, F_UPDATE_FIELDS, TH>(c, a, count, cell, out, grid);
	else switch(c.features&(F_VOLUME_FORCE|F_EQUILIBRIUM)) {
		case 0u: run_probe<P, 0u, TH>(c, a, count, cell, out, grid); break;
		case F_VOLUME_FORCE: run_probe<P, F_VOLUME_FORCE, TH>(c, a, count, cell, out, grid); break;
		case F_EQUILIBRIUM: run_probe<P, F_EQUILIBRIUM, TH>(c, a, count, cell, out, grid); break;
		default: run_probe<P, F_VOLUME_FORCE|F_EQUILIBRIUM, TH>(c, a, count, cell, out, grid); break;
	}
}
template<int P> static void pick_th(const DomainConst& c, const StepArgs& a, uint64_t count, const uint64_t* cell, float* out, unsigned grid) {
	if(c.features&F_TEMPERATURE) pick<P, true>(c, a, count, cell, out, grid); else pick<P, false>(c, a, count, cell, out, grid);
}
extern "C" int emu_probe_sample(const DomainConst* c, const StepArgs* a, uint64_t count, const uint64_t* cell, float* out, unsigned grid) {
	BY_PRECISION(*c, pick_th<P>(*c, *a, count, cell, out, grid));
	return 0;
}
'''


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not os.path.isfile("/usr/local/cuda/include/cuda_fp16.h"):
        pytest.skip("CUDA headers not installed")
    from tests.test_kernel_source_on_host import StepArgs
    d = tmp_path_factory.mktemp("probes_emu")
    src, so = d / "probes_on_host.cpp", str(d / "libprobes_emu.so")
    src.write_text(EMU_SRC)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared", "-fPIC", "-w", "-I/usr/local/cuda/include",
                           "-I" + os.path.join(ROOT, "tests", "host_emulation"), "-I" + os.path.join(ROOT, "latticeurbanwind_b200", "csrc"), str(src), "-o", so])
    L = C.CDLL(so)
    L.emu_sizeof_domain_const.restype = C.c_uint64
    L.emu_make_domain.argtypes = [C.c_void_p] + [C.c_uint32] * 6 + [C.c_int] * 4 + [C.c_uint32, C.c_float, C.c_int, C.c_uint32, C.c_float, C.c_int, C.c_uint32] + \
        [C.c_void_p] * 8 + [C.c_float] * 3
    L.emu_zone_tables.argtypes = [C.c_uint32, C.c_uint32, C.c_float, C.c_void_p, C.c_void_p]
    L.emu_probe_sample.argtypes = [C.c_void_p, C.POINTER(StepArgs), C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint]
    return L


def _cpu_case(thermal):
    """The thermal urban case (TYPE_S, TYPE_E | TYPE_T, TYPE_T sources) plus a few TYPE_G cells, on a padded row pitch (Nx = 20 -> 32)."""
    from tests import helpers as H
    flags, rho, u, T = H.thermal_case()
    flags = flags.copy()
    rng = np.random.default_rng(8)
    fluid = np.flatnonzero((flags & 0x3F) == 0)
    flags[rng.choice(fluid, 12, replace=False)] |= 0x20
    if not thermal:
        flags[(flags & 0x03) == 0] &= ~np.uint8(0x04)
    return flags, rho, u, T


@pytest.mark.parametrize("thermal", [False, True], ids=["plain", "thermal"])
@pytest.mark.parametrize("feat", FEATS)
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_kernel_source_equals_the_oracle(emu, precision, feat, thermal):
    """Every cell of the lattice plus duplicates, at an odd and an even t after oracle steps: the probe == the C oracle's update_fields read at the cell (the stored
    fields on UPDATE_FIELDS domains, at TYPE_S / TYPE_G cells and for rho / u of TYPE_E cells), bit for bit."""
    from oracle import oracle as O
    from tests import helpers as H
    from tests.test_kernel_source_on_host import HostDomain, StepArgs
    shape = H.THERMAL_SHAPE
    N = int(np.prod(shape))
    features = _features(feat, thermal)
    flags, rho0, u0, T0 = _cpu_case(thermal)
    w = cases.relaxation_rate(1e-6)
    orc = O.Oracle().bind(O.make_params(*shape, precision, features, w=w, **H.ZONES))
    fi = np.zeros(19 * N, O.ddf_dtype(precision))
    rho, u, T = rho0.copy(), u0.copy(), T0.copy()
    gi = np.zeros(7 * N, O.ddf_dtype(precision))
    if thermal:
        orc.set_thermal(**H.THERMAL)
        orc.initialize_thermal(fi, rho, u, flags, gi, T)
    else:
        orc.initialize(fi, rho, u, flags)
    rng = np.random.default_rng(precision * 100 + feat)
    cells = np.concatenate([np.arange(N), rng.choice(N, 64)]).astype(np.int64)
    Nx, Ny, _ = shape
    x, y, z = cells % Nx, (cells // Nx) % Ny, cells // (Nx * Ny)
    d = HostDomain(emu, shape, precision, features, w, H.ZONES, thermal=H.THERMAL if thermal else None)
    dev = (x + (y + z * Ny) * d.Px).astype(np.uint64)
    comps = 5 if thermal else 4
    bo = flags[cells] & 0x03
    for t in range(7):
        if thermal:
            orc.stream_collide_thermal(fi, rho, u, flags, t, H.FORCE, H.OMEGA, gi, T)
        else:
            orc.stream_collide(fi, rho, u, flags, t, H.FORCE, H.OMEGA)
        if t < 4:
            continue
        t1 = t + 1  # samples at t = 5, 6, 7: both parities
        d.put(d.fi, fi, 19); d.put(d.rho, rho, 1); d.put(d.u, u, 3); d.put(d.flags, flags, 1)
        if thermal:
            d.put(d.gi, gi, 7); d.put(d.T, T, 1)
        out = np.full(comps * cells.size, np.nan, np.float32)
        assert emu.emu_probe_sample(d.c, C.byref(StepArgs(t1, *map(np.float32, H.FORCE), *map(np.float32, H.OMEGA))), cells.size, dev.ctypes.data, out.ctypes.data, 3) == 0
        r, uu, TT = rho.copy(), u.copy(), T.copy()
        if not feat & UF:
            if thermal:
                orc.update_fields_thermal(fi, r, uu, flags, t1, H.FORCE, H.OMEGA, gi, TT)
            else:
                orc.update_fields(fi, r, uu, flags, t1, H.FORCE, H.OMEGA)
        want = [r[cells], uu[cells], uu[N + cells], uu[2 * N + cells]] + ([TT[cells]] if thermal else [])
        assert np.array_equal(_bits(out), _bits(np.concatenate(want))), t1
        # the stored fields where update_fields leaves them alone
        skip = (bo == 0x01) | ((flags[cells] & 0x38) == 0x20) | ((bo == 0x02) if feat & EQ else False) | bool(feat & UF)
        assert np.array_equal(_bits(out[:cells.size][skip]), _bits(rho[cells][skip])) and skip.any() and (~skip).any() == (not feat & UF)
        assert d.get(d.rho, 1).tobytes() == rho.tobytes() and d.get(d.u, 3).tobytes() == u.tobytes()  # nothing written into the lattice


# ---------------------------------------------------------------------------------------------------------------- CPU: ABI surface
NAMES = ("luw_probes_create", "luw_probes_sample", "luw_probes_drain", "luw_probes_reset", "luw_probes_destroy")


def test_abi_symbols_are_bound():
    from latticeurbanwind_b200 import _cabi as A
    L = A.lib()
    out = subprocess.check_output(["nm", "-D", "--defined-only", A.LIB_PATH], text=True)
    for name in NAMES:
        assert f" T {name}\n" in out + "\n" and getattr(L, name).argtypes == A.EXPORTS[name], name


def test_no_device_means_error_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    from latticeurbanwind_b200 import _cabi as A
    L = A.lib()
    cells, h, n = np.zeros(2, np.uint64), C.c_void_p(), C.c_uint64(7)
    assert L.luw_probes_create(None, 2, cells.ctypes.data, 4, C.byref(h)) == A.ERR_NO_DEVICE and not h.value
    assert L.luw_probes_sample(None, 0, *[0.0] * 6) == A.ERR_NO_DEVICE
    assert L.luw_probes_drain(None, None, C.byref(n)) == A.ERR_NO_DEVICE and n.value == 7
    assert L.luw_probes_reset(None) == A.ERR_NO_DEVICE
    assert L.luw_probes_destroy(None) == A.ERR_NO_DEVICE
    assert L.luw_last_error_string()


# ---------------------------------------------------------------------------------------------------------------- CPU: point ownership, columns
@pytest.mark.parametrize("D", [(1, 1, 1), (2, 1, 1), (1, 2, 2), (2, 2, 2)], ids=["1x1x1", "2x1x1", "1x2x2", "2x2x2"])
def test_every_point_has_exactly_one_owner(D):
    Ng, Nl, doms = split((12, 10, 8), D)
    offsets = [O for _, O in doms]
    gx, gy, gz = np.meshgrid(np.arange(Ng[0]), np.arange(Ng[1]), np.arange(Ng[2]), indexing="ij")
    pts = np.stack([gx.ravel(), gy.ravel(), gz.ravel()], axis=1)
    block, local = probe_owners(Ng, D, offsets, Nl, pts)
    gidx = pts[:, 0] + (pts[:, 1] + pts[:, 2] * Ng[1]) * Ng[0]
    H = [1 if d > 1 else 0 for d in D]
    owners = np.zeros(int(np.prod(Ng)), np.int64)
    for b, O in enumerate(offsets):
        g = _local_index(Ng, Nl, O)
        sel = block == b
        assert np.array_equal(g[local[sel]], gidx[sel])  # the local index is the point
        lx, ly, lz = local[sel] % Nl[0], (local[sel] // Nl[0]) % Nl[1], local[sel] // (Nl[0] * Nl[1])
        assert ((lx >= H[0]) & (lx < Nl[0] - H[0]) & (ly >= H[1]) & (ly < Nl[1] - H[1]) & (lz >= H[2]) & (lz < Nl[2] - H[2])).all()  # never a halo cell
        keep = np.ones(Nl[::-1], bool)
        if H[0]: keep[:, :, 0] = keep[:, :, -1] = False
        if H[1]: keep[:, 0, :] = keep[:, -1, :] = False
        if H[2]: keep[0, :, :] = keep[-1, :, :] = False
        owners += np.bincount(g[keep.reshape(-1)], minlength=owners.size)
    assert (owners == 1).all() and (block >= 0).all()
    for bad in ([12, 0, 0], [0, -1, 0], [0, 0, 8]):
        with pytest.raises(ValueError):
            probe_owners(Ng, D, offsets, Nl, [[1, 1, 1], bad])


def test_probe_columns_on_hand_made_grounds():
    g = np.array([[0, 3, 0xFFFFFFFF], [5, 1, 2]], np.uint32)  # [Ny=2][Nx=3]
    xy = [[0, 0], [1, 0], [2, 0], [0, 1], [1, 1], [2, 1]]
    pts, dropped = probe_columns(g, xy, [1, 2], 7)
    assert dropped.tolist() == [2, 3]  # no ground; 5 + 2 = 7 lies above a lattice of 7 layers
    assert pts.tolist() == [[0, 0, 1], [0, 0, 2], [1, 0, 4], [1, 0, 5], [1, 1, 2], [1, 1, 3], [2, 1, 3], [2, 1, 4]]
    pts, dropped = probe_columns(g, xy, [0], 8)
    assert dropped.tolist() == [2] and pts[:, 2].tolist() == [0, 3, 5, 1, 2]
    for bad in ([[3, 0]], [[0, 2]], [[-1, 0]]):
        with pytest.raises(ValueError):
            probe_columns(g, bad, [1], 8)


# ---------------------------------------------------------------------------------------------------------------- GPU
SMALL = dict(edge=8, pitch=16)


def _domain(shape, precision, features, arith, thermal=False):
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain
    from tests import helpers as H
    d = Domain(*shape, precision=precision, features=features, w=cases.relaxation_rate(1e-6), arith=A.ARITH_STRICT if arith == 0 else A.ARITH_FAST, **H.ZONES)
    if thermal:
        flags, rho, u, T = H.thermal_case(shape)
        d.set_thermal(**H.THERMAL)
        d.T[:] = T
    else:
        flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    d.rho[:], d.u[:], d.flags[:] = rho, u, flags
    d.f, d.omega = H.FORCE, H.OMEGA
    d.upload_all()
    d.t = 1
    d.enqueue_initialize()
    d.t = 0
    return d, flags


def _fields_at(d, cells):
    """rho / u (/ T) at the cells through a cell set, [c][k]"""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import CellSet
    cs = CellSet(d, cells)
    r, u = np.empty(cells.size, np.float32), np.empty(3 * cells.size, np.float32)
    cs.download(A.FIELD_RHO, r)
    cs.download(A.FIELD_U, u)
    parts = [r, u]
    if d.thermal:
        T = np.empty(cells.size, np.float32)
        cs.download(A.FIELD_T, T)
        parts.append(T)
    d.finish_queue()
    cs.close()
    return np.concatenate(parts).reshape(-1, cells.size)


def _cells(shape, seed=3, k=3000):
    rng = np.random.default_rng(seed)
    N = int(np.prod(shape))
    return np.concatenate([rng.choice(N, k, replace=False), rng.choice(N, 16)]).astype(np.uint64)  # with duplicates


def _check_against_update_fields(d, pr, cells, feat):
    """sample() leaves the fields alone and equals update_fields + cell-set download (UPDATE_FIELDS domains: the stored fields), bit for bit."""
    before = _fields_at(d, cells)
    pr.sample()
    got = pr.drain()
    assert got.shape == (1, 5 if d.thermal else 4, cells.size)
    assert np.array_equal(_bits(_fields_at(d, cells)), _bits(before))  # no side effect
    if not feat & UF:
        d.enqueue_update_fields()
    want = _fields_at(d, cells)
    assert np.array_equal(_bits(got[0]), _bits(want))
    return got[0]


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("Nx", [63, 64], ids=["padded", "dense"])
@pytest.mark.parametrize("feat", FEATS)
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_sample_equals_update_fields(precision, feat, Nx, arith):
    """After 3 and after 4 steps (odd and even t): sample == luw_update_fields + cell-set download on the same domain, bit for bit; the fields are unchanged
    by sample."""
    from latticeurbanwind_b200.domain import Probes
    shape = (Nx, 48, 32)
    d, flags = _domain(shape, precision, _features(feat), arith)
    cells = _cells(shape)
    with d:
        pr = Probes(d, cells, 4)
        d.run_steps(3)
        a = _check_against_update_fields(d, pr, cells, feat)
        d.run_steps(1)
        b = _check_against_update_fields(d, pr, cells, feat)
        assert not np.array_equal(a, b) and np.isfinite(b).all()
        assert ((flags[cells.astype(np.int64)] & 3) == 1).any() and ((flags[cells.astype(np.int64)] & 3) == 2).any()
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("feat", [14, 15])
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_thermal_sample_equals_update_fields_thermal(precision, feat, arith):
    """LUW_TEMPERATURE domains: rho / u / T == update_fields_thermal + cell-set download (FEAT 15: the stored fields), bit for bit, no side effect."""
    from latticeurbanwind_b200.domain import Probes
    shape = (36, 32, 20)
    d, _ = _domain(shape, precision, _features(feat, True), arith, thermal=True)
    cells = _cells(shape, k=2000)
    with d:
        pr = Probes(d, cells, 2)
        for steps in (3, 1):
            d.run_steps(steps)
            got = _check_against_update_fields(d, pr, cells, feat)
            assert np.isfinite(got).all() and got[4].std() > 0
        pr.close()


def _oracle_series(shape, precision, features, steps, cells):
    """rho / u after update_fields at t = 1..steps on the C oracle (STRICT arithmetic), at the cells: [steps][4][k]."""
    from oracle import oracle as O
    from tests import helpers as H
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    N = int(np.prod(shape))
    orc = O.Oracle().bind(O.make_params(*shape, precision, features, w=cases.relaxation_rate(1e-6), **H.ZONES))
    fi = np.zeros(19 * N, O.ddf_dtype(precision))
    rho, u = rho.copy(), u.copy()
    orc.initialize(fi, rho, u, flags)
    out = []
    for t in range(steps):
        orc.stream_collide(fi, rho, u, flags, t, H.FORCE, H.OMEGA)
        r, uu = rho.copy(), u.copy()
        orc.update_fields(fi, r, uu, flags, t + 1, H.FORCE, H.OMEGA)
        c = cells.astype(np.int64)
        out.append(np.stack([r[c], uu[c], uu[N + c], uu[2 * N + c]]))
    return np.stack(out)


def _lbm(shape, D, precision, features, arith):
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import LBM
    from tests import helpers as H
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    lbm = LBM(shape, D=D, precision=precision, features=features, arith=A.ARITH_STRICT if arith == 0 else A.ARITH_FAST, nu=1e-6, f=H.FORCE, omega=H.OMEGA,
              **H.ZONES)
    lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
    lbm.run(0)
    return lbm


def _points(shape, P=500, seed=9):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(0, n, P) for n in shape], axis=1)


def _lbm_series(shape, D, precision, features, arith, steps, points, capacity=256):
    from latticeurbanwind_b200.lbm import Probes
    lbm = _lbm(shape, D, precision, features, arith)
    pr = Probes(lbm, points, capacity)
    for _ in range(steps):
        lbm.run(1)
        pr.sample()
    s = pr.series()
    pr.close()
    lbm.close()
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_strict_series_equal_the_c_oracle(precision):
    shape = (48, 40, 32)
    pts = _points(shape)
    feat = _features(14)
    s = _lbm_series(shape, (1, 1, 1), precision, feat, 0, 5, pts)
    cells = (pts[:, 0] + (pts[:, 1] + pts[:, 2] * shape[1]) * shape[0]).astype(np.uint64)
    want = _oracle_series(shape, precision, feat, 5, cells)
    assert s["t"].tolist() == [1, 2, 3, 4, 5] and s["rho"].shape == (5, pts.shape[0]) and s["u"].shape == (5, 3, pts.shape[0]) and "T" not in s
    assert np.array_equal(_bits(s["rho"]), _bits(want[:, 0])) and np.array_equal(_bits(s["u"]), _bits(want[:, 1:]))


@pytest.mark.gpu
def test_stream_order_with_automatic_drains():
    """40 steps with a sample after each and no synchronisation in between == update_fields + download after every step; the same through lbm.Probes with
    capacity 16, whose ring drains itself when full."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Probes
    shape = (64, 48, 32)
    feat = _features(14)
    d, _ = _domain(shape, A.FP16S, feat, 1)
    cells = _cells(shape, k=1000)
    with d:
        pr = Probes(d, cells, 40)
        for s in range(40):
            d.run_steps(1)
            pr.sample()
        got = pr.drain()
        pr.close()
    ref = []
    d, _ = _domain(shape, A.FP16S, feat, 1)
    with d:
        for s in range(40):
            d.run_steps(1)
            d.enqueue_update_fields()
            ref.append(_fields_at(d, cells))
    assert got.shape == (40, 4, cells.size) and np.array_equal(_bits(got), _bits(np.stack(ref)))
    # the same through lbm.Probes, which drains when its ring is full
    pts = np.stack([cells.astype(np.int64) % 64, (cells.astype(np.int64) // 64) % 48, cells.astype(np.int64) // (64 * 48)], axis=1)
    s = _lbm_series(shape, (1, 1, 1), A.FP16S, feat, 1, 40, pts, capacity=16)
    assert s["t"].tolist() == list(range(1, 41))
    assert np.array_equal(_bits(s["rho"]), _bits(got[:, 0])) and np.array_equal(_bits(s["u"]), _bits(got[:, 1:4]))


@pytest.mark.gpu
def test_ring_full_drain_order_reset_and_invalid_arguments():
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, Probes
    Lib = A.lib()
    shape = (64, 48, 32)
    d, _ = _domain(shape, A.FP32, _features(14), 0)
    cells = _cells(shape, k=100)
    with d:
        pr = Probes(d, cells, 3)
        for _ in range(3):
            d.run_steps(1)
            pr.sample()
        assert Lib.luw_probes_sample(pr._h, d.t, *[0.0] * 6) == A.ERR_INVALID  # ring full
        got = pr.drain()
        assert got.shape == (3, 4, cells.size) and pr.drain().shape[0] == 0
        assert not np.array_equal(got[0], got[1]) and not np.array_equal(got[1], got[2])
        pr.sample(t=d.t)
        last = pr.drain()[0]
        assert np.array_equal(_bits(last), _bits(got[2]))  # drain order: the last sample of the ring is the current state
        pr.sample()
        pr.reset()
        assert pr.drain().shape[0] == 0
        d.finish_queue()
        n0 = d.launch_count()
        pr.sample()
        assert d.launch_count() == n0 + 1  # one kernel per sample
        pr.close()
        empty = Probes(d, np.zeros(0, np.uint64), 2)  # count 0
        empty.sample(); empty.sample()
        assert empty.drain().shape == (2, 4, 0)
        empty.close()
        h = C.c_void_p()

        def create(cells=cells[:2], cap=4, null_list=False, count=None):
            c = np.ascontiguousarray(cells, np.uint64)
            return Lib.luw_probes_create(d._h, c.size if count is None else count, None if null_list else c.ctypes.data, cap, C.byref(h))
        assert create() == A.OK
        Lib.luw_probes_destroy(h)
        for kw in (dict(cells=[d.N]), dict(null_list=True), dict(cap=0)):
            h = C.c_void_p()
            assert create(**kw) == A.ERR_INVALID and not h.value, kw
    # halo indices are rejected on a decomposed block
    with Domain(34, 24, 16, D=(2, 1, 1), O=(-1, 0, 0), precision=A.FP32, features=0, w=1.0) as d:
        for cell in (0, 33, 1 + 34, 34 * 24 * 16 - 1):
            h = C.c_void_p()
            cl = np.array([cell], np.uint64)
            assert Lib.luw_probes_create(d._h, 1, cl.ctypes.data, 1, C.byref(h)) == (A.OK if cell == 35 else A.ERR_INVALID), cell
            Lib.luw_probes_destroy(h)


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("D", [(2, 1, 1), (1, 2, 2), (2, 2, 2)], ids=["2x1x1", "1x2x2", "2x2x2"])
def test_decompositions_equal_the_single_domain(D, arith):
    """In-process decompositions give the single domain's series bit for bit. Nx = 256 keeps every block at least 128 cells wide, so that in FAST every block
    runs the same step kernel as the single domain (a block narrower than the 128-wide tiles takes another FAST step kernel, whose DDFs differ in the last bits)."""
    from latticeurbanwind_b200 import _cabi as A
    shape = (256, 48, 32)
    pts = _points(shape, P=800)
    feat = _features(14)
    one = _lbm_series(shape, (1, 1, 1), A.FP16S, feat, arith, 5, pts, capacity=2)
    dec = _lbm_series(shape, D, A.FP16S, feat, arith, 5, pts, capacity=2)
    for k in ("t", "rho", "u"):
        assert np.array_equal(np.asarray(one[k]).view(np.uint8), np.asarray(dec[k]).view(np.uint8)), k


@pytest.mark.gpu
def test_cpp_host_layer_equals_the_python_path(tmp_path):
    """LBM_Probes (C++ host layer, through luw_host_case's LUW_CASE_PROBES switch) == lbm.Probes on the same case, single domain and [1,2,2]."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import Probes
    from tests import helpers as H
    from tests.test_cpp_host import build, run_driver
    build()
    shape, steps, samples = (64, 48, 32), 7, 5
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    feat = _features(14)
    pts = _points(shape, P=300)
    for D in ((1, 1, 1), (1, 2, 2)):
        path = str(tmp_path / "probes.bin")
        env_keep = dict(os.environ)
        os.environ.update(LUW_CASE_PROBES=",".join(str(v) for v in pts.reshape(-1)), LUW_CASE_PROBES_OUT=path, LUW_CASE_PROBES_CAP="2")
        try:
            run_driver(tmp_path, shape, D, A.FP16S, feat, 0, 1e-6, steps, flags, rho, u, zones=H.ZONES, stats=samples)
        finally:
            os.environ.clear()
            os.environ.update(env_keep)
        raw = open(path, "rb").read()
        n, comps, P = int(np.frombuffer(raw[:8], np.uint64)[0]), int(np.frombuffer(raw[8:12], np.uint32)[0]), int(np.frombuffer(raw[12:20], np.uint64)[0])
        t = np.frombuffer(raw[20:20 + 8 * n], np.uint64)
        vals = np.frombuffer(raw[20 + 8 * n:], np.float32).reshape(n, comps, P)
        lbm = _lbm(shape, D, A.FP16S, feat, 0)
        lbm.run(steps - samples)
        pr = Probes(lbm, pts, 2)
        for _ in range(samples):
            lbm.run(1)
            pr.sample()
        s = pr.series()
        assert n == samples and comps == 4 and P == pts.shape[0]
        assert t.tolist() == s["t"].tolist() == list(range(steps - samples + 1, steps + 1))
        assert np.array_equal(_bits(vals[:, 0]), _bits(s["rho"])) and np.array_equal(_bits(vals[:, 1:]), _bits(s["u"])), D
        pr.close()
        lbm.close()
