"""Wind loads on buildings (csrc/lbm_wall_loads.cuh, luw_solid_surface, luw_wall_loads_*, domain.WallLoads, lbm.WallLoads, LBM_WallLoads).
CPU: the oracle on hand-made lattices and on a Poiseuille channel run by the C oracle (momentum balance); the kernel source compiled for host threads against
the oracle; the ABI surface. GPU: the device path against the oracle on the downloaded DDFs, the momentum balance, decompositions, stream order and error
paths, and the C++ host layer. Bar: bit for bit, except label sums against math.fsum and across decompositions (1e-12 relative)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from latticeurbanwind_b200 import cases
from oracle import wall_loads_oracle as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPE_S, TYPE_E = 0x01, 0x02


# ---------------------------------------------------------------------------------------------------------------- CPU: oracle on hand-made lattices
def _store(shape, n, f, odd):
    """Dense FP32 DDF image whose load_f at cell n returns f[19] (Esoteric-Pull: f[i] of odd i sits in slot i (odd t) / i+1 (even t) at n, f[i+1] in slot
    i+1 / i at n + c_i)."""
    Nx, Ny, Nz = shape
    N = Nx * Ny * Nz
    fi = np.zeros(19 * N, np.float32)
    x, y, z = n % Nx, (n // Nx) % Ny, n // (Nx * Ny)
    fi[n] = f[0]
    for i in range(1, 19, 2):
        j = (x + W.CX[i]) % Nx + ((y + W.CY[i]) % Ny + ((z + W.CZ[i]) % Nz) * Ny) * Nx
        fi[(i if odd else i + 1) * N + n] = f[i]
        fi[(i + 1 if odd else i) * N + j] = f[i + 1]
    return fi


@pytest.mark.parametrize("odd", [0, 1])
def test_single_solid_cell_force_by_hand(odd):
    """One solid cell in a periodic box: every link counts and F = 2 sum_i c_i f_i, here with dyadic f_i so that the hand sum is exact."""
    shape = (5, 5, 5)
    flags = np.zeros(125, np.uint8)
    n = 2 + (2 + 2 * 5) * 5
    flags[n] = TYPE_S
    cells, m = W.surface(flags, shape, (True, True, True))
    assert cells.tolist() == [n] and m[0] == (1 << 19) - 2
    f = (np.arange(19) * 2.0 ** -7 - 2.0 ** -4).astype(np.float32)
    F = W.cell_forces(W.load_f(_store(shape, n, f, odd), shape, 0, cells, odd), m)
    hand = [2.0 * sum(float(c[i]) * float(f[i]) for i in range(19)) for c in (W.CX, W.CY, W.CZ)]
    assert F[:, 0].tolist() == hand and any(hand)
    M = W.moments(F, [2], [2], [2], [[0.0, 0.0, 0.5]])
    assert M[:, 0].tolist() == [2.0 * hand[2] - 1.5 * hand[1], 1.5 * hand[0] - 2.0 * hand[2], 2.0 * hand[1] - 2.0 * hand[0]]


def _ground_plane(top=0):
    shape = (4, 3, 4)
    f = np.zeros((4, 3, 4), np.uint8)
    f[0] = TYPE_S
    f[3] = top
    return f.reshape(-1), shape


UP = sum(1 << i for i in range(19) if W.CZ[i] == -1)  # partner n - c_i one layer up
DOWN = sum(1 << i for i in range(19) if W.CZ[i] == 1)  # partner one layer down: across z = 0


def test_wall_at_a_non_periodic_face_excludes_wrap_links():
    flags, shape = _ground_plane()
    cells, m = W.surface(flags, shape, (True, True, False))
    assert cells.tolist() == list(range(12)) and (m == UP).all()  # in-plane partners are solid, the wrap to z = 3 crosses the face


def test_wall_links_count_once_the_axis_is_periodic():
    flags, shape = _ground_plane()
    cells, m = W.surface(flags, shape, (True, True, True))
    assert cells.tolist() == list(range(12)) and (m == UP | DOWN).all()
    # a solid top layer closes the wrap again (and is a wall itself), and a lattice that is solid throughout lists nothing
    flags2, _ = _ground_plane(top=TYPE_S)
    cells, m = W.surface(flags2, shape, (True, True, True))
    assert cells.tolist() == list(range(12)) + list(range(36, 48)) and (m[:12] == UP).all() and (m[12:] == DOWN).all()
    assert W.surface(np.full(48, TYPE_S, np.uint8), shape, (True, True, True))[0].size == 0


def test_type_e_partners_count():
    flags, shape = _ground_plane(top=TYPE_E | 0x04)
    _, m = W.surface(flags, shape, (True, True, True))
    assert (m == UP | DOWN).all()
    _, m = W.surface(flags, shape, (True, True, False))
    assert (m == UP).all()


def test_footprint_labels_and_reference_points():
    """Two footprints that touch along an edge are one building; a diagonal contact is not 4-connected; numbering follows the first column in (y, x) order."""
    from latticeurbanwind_b200.lbm import footprint_labels, footprint_ref_points
    g = np.ones((6, 8), np.uint32)
    g[0:2, 5:7] = 4  # B: first in row-major order
    g[1:3, 1:3] = 3  # A, touching A2 along an edge
    g[3, 1:4] = 0xFFFFFFFF  # A2 (all solid columns count as building)
    g[4, 4] = 2  # a one-column building (ground 2 > ground_z + 1) touching A2 only diagonally: its own label
    want = np.zeros((6, 8), np.uint32)
    want[0:2, 5:7] = 1
    want[1:3, 1:3] = 2
    want[3, 1:4] = 2
    want[4, 4] = 3
    for fn in (W.footprint_labels, footprint_labels):
        assert np.array_equal(fn(g, 0), want)
    assert not W.footprint_labels(g, 1)[4, 4]  # with ground_z = 1 a ground of 2 is terrain
    r0 = W.ref_points(want, 4, 0)
    assert r0.tolist() == [[0, 0, 0], [5.5, 0.5, 0.5], [(1 + 2 + 1 + 2 + 1 + 2 + 3) / 7, (1 + 1 + 2 + 2 + 3 + 3 + 3) / 7, 0.5], [4.0, 4.0, 0.5]]
    assert np.array_equal(footprint_ref_points(want, 4, 0), r0)
    assert W.cell_labels([5, 5, 4], [0, 0, 4], [1, 0, 3], want).tolist() == [1, 0, 3]


def test_label_sums_two_level_order_against_fsum():
    rng = np.random.default_rng(5)
    K, L = 200, 4
    labels = np.sort(rng.integers(0, L - 1, K)).astype(np.uint32)  # label 3 has no cells
    F = rng.standard_normal((3, K)).astype(np.float32)
    M = rng.standard_normal((3, K)) * 100
    got = W.label_sums(F, M, labels, L)
    V = np.concatenate([F.astype(np.float64), M])
    for l in range(L):
        for a in range(6):
            ref = math.fsum(V[a, labels == l])
            assert abs(got[l, a] - ref) <= 1e-12 * max(abs(ref), 1.0)
    assert not got[3].any()


def poiseuille(steps=1920):
    """Plane Poiseuille channel on the C oracle: 4 x 4 x 10, walls at z = 0 and 9, FP32, VOLUME_FORCE only, tau = 1 (nu = 1/6): 5 diffusion times H^2/nu
    for H = 8. Returns (fi, flags, shape, fx, fluid cells)."""
    from oracle import oracle as O
    shape = (4, 4, 10)
    N = int(np.prod(shape))
    flags = np.zeros((10, 4, 4), np.uint8)
    flags[0] = flags[-1] = TYPE_S
    flags = flags.reshape(-1)
    rho, u = np.ones(N, np.float32), np.zeros(3 * N, np.float32)
    fx = 1e-5
    orc = O.Oracle().bind(O.make_params(*shape, O.FP32, O.VOLUME_FORCE, w=1.0))
    fi = np.zeros(19 * N, np.float32)
    orc.initialize(fi, rho, u, flags)
    for t in range(steps):
        orc.stream_collide(fi, rho, u, flags, t, (fx, 0.0, 0.0), (0.0, 0.0, 0.0))
    return fi, flags, shape, fx, 8 * 16


def check_balance(F, z, Nz, fx, fluid):
    """Sum of Fx over both walls == fx x fluid cells within 1e-3, each wall (its own label) half of it; no net normal or cross-stream load."""
    want = fx * fluid
    per = [math.fsum(F[0][z == zz].astype(np.float64)) for zz in (0, Nz - 1)]
    assert abs(sum(per) - want) <= 1e-3 * want, (per, want)
    for p in per:
        assert abs(p - want / 2) <= 1e-3 * want / 2, (per, want)
    assert abs(math.fsum(F[1].astype(np.float64))) <= 1e-6 * want


def test_momentum_balance_in_the_c_oracle():
    fi, flags, shape, fx, fluid = poiseuille()
    cells, m = W.surface(flags, shape, (True, True, False))
    assert cells.size == 32
    z = cells.astype(np.int64) // 16
    F = W.cell_forces(W.load_f(fi, shape, 0, cells, 1920 % 2), m)  # the state after 1920 steps is read with t = 1920
    check_balance(F, z, shape[2], fx, fluid)
    L2 = W.label_sums(F, np.zeros((3, cells.size)), (z > 0).astype(np.uint32), 2)  # each wall its own label
    assert abs(L2[0, 0] - L2[1, 0]) <= 1e-3 * fx * fluid and abs(L2[0, 0] + L2[1, 0] - fx * fluid) <= 1e-3 * fx * fluid


# ---------------------------------------------------------------------------------------------------------------- CPU: kernel source on host threads
EMU_SRC = r'''
#include "cuda_on_host.hpp"
static inline double __dadd_rn(double a, double b) { return a+b; }
static inline double __dsub_rn(double a, double b) { return a-b; }
static inline double __dmul_rn(double a, double b) { return a*b; }
#include "lbm_wall_loads.cuh"
static luw::DomainConst dc(uint32_t Nx, uint32_t Ny, uint32_t Nz, uint32_t Px, int precision, void* fi, uint8_t* flags) {
	luw::DomainConst c; memset(&c, 0, sizeof(c));
	c.Nx = Nx; c.Ny = Ny; c.Nz = Nz; c.Px = Px; c.N = (uint64_t)Px*Ny*Nz; c.Dx = c.Dy = c.Dz = 1u; c.Nxg = Nx; c.Nyg = Ny; c.Nzg = Nz;
	c.precision = precision; c.fi = fi; c.flags = flags;
	return c;
}
#define EMU_LAUNCH(grid, call) { emu_blockDim = {256u, 1u, 1u}; emu_gridDim = {(unsigned)(grid), 1u, 1u}; \
	for(unsigned b=0u; b<(unsigned)(grid); b++) for(unsigned i=0u; i<256u; i++) { emu_blockIdx = {b, 0u, 0u}; emu_threadIdx = {i, 0u, 0u}; call; } }
extern "C" {
void emu_surface(uint32_t Nx, uint32_t Ny, uint32_t Nz, uint32_t Px, uint8_t* flags, uint32_t periodic, const uint64_t* offset, uint32_t* count, uint64_t* cells, unsigned grid) {
	const luw::DomainConst c = dc(Nx, Ny, Nz, Px, 0, nullptr, flags);
	EMU_LAUNCH(grid, luw::k_surface_rows(c, periodic, 0u, Nx, 0u, Ny, 0u, Nz, offset, count, cells));
}
void emu_links(uint32_t Nx, uint32_t Ny, uint32_t Nz, uint32_t Px, uint8_t* flags, uint32_t periodic, uint64_t count, const uint64_t* cell, uint32_t* links, unsigned grid) {
	const luw::DomainConst c = dc(Nx, Ny, Nz, Px, 0, nullptr, flags);
	EMU_LAUNCH(grid, luw::k_wall_links(c, periodic, count, cell, links));
}
void emu_cells(uint32_t Nx, uint32_t Ny, uint32_t Nz, uint32_t Px, int precision, void* fi, uint64_t count, const uint64_t* cell, const uint32_t* links, uint32_t odd,
	float inv_n, float* F, float* acc, unsigned grid) {
	const luw::DomainConst c = dc(Nx, Ny, Nz, Px, precision, fi, nullptr);
	if(precision==0) EMU_LAUNCH(grid, luw::k_wall_cells<0>(c, count, cell, links, odd, inv_n, F, acc))
	else if(precision==1) EMU_LAUNCH(grid, luw::k_wall_cells<1>(c, count, cell, links, odd, inv_n, F, acc))
	else EMU_LAUNCH(grid, luw::k_wall_cells<2>(c, count, cell, links, odd, inv_n, F, acc))
}
void emu_reduce(uint32_t Nx, uint32_t Ny, uint32_t Nz, uint32_t Px, uint64_t count, uint64_t nchunks, const uint64_t* chunk_begin, const uint32_t* chunk_label,
	const uint64_t* cell, const float* F, const double* ref, double* partial, uint64_t ngroups, const uint64_t* group_begin, double* partial2, uint32_t L,
	const uint64_t* label_group, double* out, unsigned grid) {
	const luw::DomainConst c = dc(Nx, Ny, Nz, Px, 0, nullptr, nullptr);
	EMU_LAUNCH(grid, luw::k_wall_chunks(c, count, nchunks, chunk_begin, chunk_label, cell, F, ref, partial));
	EMU_LAUNCH(grid, luw::k_wall_segments(ngroups, group_begin, nchunks, partial, 1u, ngroups, partial2));
	EMU_LAUNCH(grid, luw::k_wall_segments(L, label_group, ngroups, partial2, 6u, 1u, out));
}
}
'''


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not os.path.isfile("/usr/local/cuda/include/cuda_fp16.h"):
        pytest.skip("CUDA headers not installed")
    d = tmp_path_factory.mktemp("wall_emu")
    src, so = d / "wall_on_host.cpp", str(d / "libwall_emu.so")
    src.write_text(EMU_SRC)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-w", "-I/usr/local/cuda/include",
                           "-I" + os.path.join(ROOT, "tests", "host_emulation"), "-I" + os.path.join(ROOT, "latticeurbanwind_b200", "csrc"), str(src), "-o", so])
    L = C.CDLL(so)
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    L.emu_surface.argtypes = [u32] * 4 + [vp, u32, vp, vp, vp, C.c_uint]
    L.emu_links.argtypes = [u32] * 4 + [vp, u32, u64, vp, vp, C.c_uint]
    L.emu_cells.argtypes = [u32] * 4 + [C.c_int, vp, u64, vp, vp, u32, C.c_float, vp, vp, C.c_uint]
    L.emu_reduce.argtypes = [u32] * 4 + [u64, u64, vp, vp, vp, vp, vp, vp, u64, vp, vp, u32, vp, vp, C.c_uint]
    return L


def _segments(labels, L, size):
    """(begin [n + 1], segment label, label_segment [L + 1]): consecutive runs of up to `size` items of one label, as luw_wall_loads_create cuts them."""
    labels = np.asarray(labels, np.int64)
    begin, lab = [], []
    for k in range(labels.size):
        if k == 0 or labels[k] != labels[k - 1] or k - begin[-1] == size:
            begin.append(k)
            lab.append(labels[k])
    lab = np.array(lab, np.int64)
    return np.array(begin + [labels.size], np.uint64), lab.astype(np.uint32), np.searchsorted(lab, np.arange(L + 1), side="left").astype(np.uint64)


def emu_reduce(emu, shape, Px, cells_dev, F, labels, ref, grid=2):
    """Host-thread run of k_wall_chunks + the two k_wall_segments levels -> float64 [L, 6]."""
    L = ref.shape[0]
    cb, cl, _ = _segments(labels, L, W.CHUNK)
    gb, _, lg = _segments(cl, L, W.GROUP)
    nch, ngr = cl.size, gb.size - 1
    partial, partial2 = np.zeros(6 * max(nch, 1), np.float64), np.zeros(6 * max(ngr, 1), np.float64)
    out = np.zeros((L, 6), np.float64)
    F = np.ascontiguousarray(F, np.float32)
    ref = np.ascontiguousarray(ref, np.float64)
    emu.emu_reduce(*shape, Px, cells_dev.size, nch, cb.ctypes.data, cl.ctypes.data, cells_dev.ctypes.data, F.ctypes.data, ref.ctypes.data, partial.ctypes.data,
                   ngr, gb.ctypes.data, partial2.ctypes.data, L, lg.ctypes.data, out.ctypes.data, grid)
    return out


def _pitched(a, shape, Px, comps):
    Nx, Ny, Nz = shape
    out = np.zeros((comps, Nz, Ny, Px), a.dtype)
    out[..., :Nx] = a.reshape(comps, Nz, Ny, Nx)
    return out


def _random_ddfs(rng, N, precision):
    if precision == 0:
        return (rng.standard_normal(19 * N) * 0.02).astype(np.float32)
    h = rng.integers(0, 65536, 19 * N).astype(np.uint16)
    if precision == 1:  # finite binary16 codes only
        h = np.where((h & 0x7C00) == 0x7C00, h & 0x83FF, h).astype(np.uint16)
    return h


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_kernel_source_equals_the_oracle(emu, precision):
    """Surface enumeration, link masks, per-cell force + Welford at even and odd t, and the two-level reduction, run on host threads over a padded-row
    urban lattice (Px = 16 > Nx = 13) == the oracle bit for bit."""
    rng = np.random.default_rng(11 + precision)
    shape, Px = (13, 11, 12), 16
    Nx, Ny, Nz = shape
    N = Nx * Ny * Nz
    flags = cases.urban(*shape, seed=4, edge=3, pitch=5)[0].copy()
    flags.reshape(Nz, Ny, Nx)[5:7, 2:4, 9:12] = TYPE_S  # an overhang
    pf = _pitched(flags, shape, Px, 1).reshape(-1)
    for periodic in ((False, False, False), (True, True, True), (True, False, True)):
        mask = sum(1 << a for a in range(3) if periodic[a])
        want, wlinks = W.surface(flags, shape, periodic)
        rows = Ny * Nz
        count = np.zeros(rows, np.uint32)
        emu.emu_surface(*shape, Px, pf.ctypes.data, mask, None, count.ctypes.data, None, 3)
        offset = np.concatenate([[0], np.cumsum(count.astype(np.uint64))[:-1]]).astype(np.uint64)
        got = np.zeros(int(count.sum()), np.uint64)
        emu.emu_surface(*shape, Px, pf.ctypes.data, mask, offset.ctypes.data, count.ctypes.data, got.ctypes.data, 3)
        assert np.array_equal(got, want), periodic
    # per-cell kernels and the reduction (non-periodic, as LUW's decks)
    cells, m = W.surface(flags, shape)
    x, y, z = cells.astype(np.int64) % Nx, (cells.astype(np.int64) // Nx) % Ny, cells.astype(np.int64) // (Nx * Ny)
    col = W.footprint_labels(W.column_ground(flags, shape), 0)
    L = int(col.max()) + 1
    labels = W.cell_labels(x, y, z, col)
    order = np.lexsort((cells, labels))
    cells, m, labels, x, y, z = cells[order], m[order], labels[order], x[order], y[order], z[order]
    dev = (x + (y + z * Ny) * Px).astype(np.uint64)
    links = np.zeros(cells.size, np.uint32)
    emu.emu_links(*shape, Px, pf.ctypes.data, 0, cells.size, dev.ctypes.data, links.ctypes.data, 2)
    assert np.array_equal(links, m)
    ref = W.ref_points(col, L)
    K = cells.size
    acc = np.zeros((6, K), np.float32)
    F = np.zeros((3, K), np.float32)
    orc = W.WelfordF(K)
    for s, t in enumerate((4, 7, 10)):  # even, odd, even
        fi = _random_ddfs(rng, N, precision)
        fp = _pitched(fi, shape, Px, 19).reshape(-1)
        inv_n = np.float32(1.0) / np.float32(s + 1)
        emu.emu_cells(*shape, Px, precision, fp.ctypes.data, K, dev.ctypes.data, links.ctypes.data, t & 1, float(inv_n), F.ctypes.data, acc.ctypes.data, 2)
        want_F = W.cell_forces(W.load_f(fi, shape, precision, cells, t & 1), m)
        assert np.array_equal(F, want_F), t
        orc.accumulate(want_F)
        assert np.array_equal(acc[:3], orc.mean) and np.array_equal(acc[3:], orc.m2), t
        M = W.moments(want_F, x, y, z, ref[labels])
        assert np.array_equal(emu_reduce(emu, shape, Px, dev, F, labels, ref), W.label_sums(want_F, M, labels, L)), t
    assert L > 2 and (labels == 0).any() and np.abs(F).max() > 0


def test_kernel_source_reduction_over_many_groups(emu):
    """The three summation levels on a list long enough for several groups per label (and a label without cells) == the oracle bit for bit."""
    rng = np.random.default_rng(3)
    shape, Px = (40, 30, 20), 48
    K, L = 9000, 5
    cells = np.sort(rng.choice(np.prod(shape), K, replace=False)).astype(np.int64)
    labels = np.sort(rng.choice([0, 0, 0, 1, 3, 4], K)).astype(np.uint32)  # label 2 empty; label 0 ~4500 cells = 141 chunks = 5 groups
    order = np.lexsort((cells, labels))
    cells, labels = cells[order], labels[order]
    x, y, z = cells % 40, (cells // 40) % 30, cells // 1200
    F = (rng.standard_normal((3, K)) * 1e-3).astype(np.float32)
    ref = rng.uniform(0, 30, (L, 3))
    dev = (x + (y + z * 30) * Px).astype(np.uint64)
    want = W.label_sums(F, W.moments(F, x, y, z, ref[labels]), labels, L)
    assert np.array_equal(emu_reduce(emu, shape, Px, dev, F, labels, ref, grid=3), want) and not want[2].any()


# ---------------------------------------------------------------------------------------------------------------- CPU: ABI surface
NAMES = ("luw_solid_surface", "luw_wall_loads_create", "luw_wall_loads_accumulate", "luw_wall_loads_drain", "luw_wall_loads_download_cells",
         "luw_wall_loads_reset", "luw_wall_loads_destroy")


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
    n = C.c_uint64(7)
    assert L.luw_solid_surface(None, 0, 0, None, C.byref(n)) == A.ERR_NO_DEVICE
    cells, labels, ref = np.zeros(2, np.uint64), np.zeros(2, np.uint32), np.zeros(3, np.float64)
    h = C.c_void_p()
    assert L.luw_wall_loads_create(None, 2, cells.ctypes.data, labels.ctypes.data, 1, ref.ctypes.data, 0, 4, C.byref(h)) == A.ERR_NO_DEVICE and not h.value
    assert L.luw_last_error_string()


# ---------------------------------------------------------------------------------------------------------------- GPU
SMALL = dict(edge=8, pitch=16)  # cases.urban(64, 48, 32, ...): 9 footprints


def _close(a, b, rel=1e-12, floor=1e-15):
    return np.all(np.abs(a - b) <= rel * np.abs(b) + floor)


def _fsum_loads(F, M, labels, L):
    V = np.concatenate([F.astype(np.float64), M])
    return np.array([[math.fsum(V[a, labels == l]) for a in range(6)] for l in range(L)])


def _labelled_list(flags, shape, ground_z=0):
    Nx, Ny, _ = shape
    cells, m = W.surface(flags, shape)
    c = cells.astype(np.int64)
    x, y, z = c % Nx, (c // Nx) % Ny, c // (Nx * Ny)
    col = W.footprint_labels(W.column_ground(flags, shape), ground_z)
    L = int(col.max()) + 1
    labels = W.cell_labels(x, y, z, col, ground_z)
    order = np.lexsort((cells, labels))
    return cells[order], m[order], labels[order], (x[order], y[order], z[order]), L, W.ref_points(col, L, ground_z)


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("Nx", [63, 64], ids=["padded", "dense"])
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_device_equals_oracle_on_urban_case(precision, Nx, arith):
    """Per sample (t = 1..4: odd and even) the label loads == the oracle's two-level sums on the downloaded DDFs bit for bit and math.fsum within 1e-12; after
    one sample the per-cell mean is F itself, after four the mean / M2 == the oracle's Welford; the list == the oracle's surface."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, WallLoads
    from tests import helpers as H
    shape = (Nx, 48, 32)
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    with Domain(*shape, precision=precision, features=H.FEATURE_SETS["luw"], w=cases.relaxation_rate(1e-6), arith=A.ARITH_STRICT if arith == 0 else A.ARITH_FAST,
                **H.ZONES) as d:
        d.rho[:], d.u[:], d.flags[:] = rho, u, flags
        d.f, d.omega = H.FORCE, H.OMEGA
        d.upload_all()
        d.t = 1
        d.enqueue_initialize()
        d.t = 0
        d.finish_queue()
        cells, m, labels, (x, y, z), L, ref = _labelled_list(flags, shape)
        assert np.array_equal(np.sort(d.solid_surface(0)), np.sort(cells)) and L == 10
        wl = WallLoads(d, cells, labels, L, ref, 0, 8)
        orc = W.WelfordF(cells.size)
        for s in range(4):
            d.enqueue_stream_collide()
            d.increment_time_step()
            wl.accumulate()
            F = W.cell_forces(W.load_f(d.read_fi(), shape, precision, cells, d.t & 1), m)
            orc.accumulate(F)
            got = wl.drain()
            assert got.shape == (1, L, 6)
            M = W.moments(F, x, y, z, ref[labels])
            assert np.array_equal(got[0], W.label_sums(F, M, labels, L)), s
            assert _close(got[0], _fsum_loads(F, M, labels, L)), s
            if s == 0:
                mean, _, n = wl.download_cells()
                assert n == 1 and np.array_equal(mean, F)
        mean, m2, n = wl.download_cells()
        assert n == 4 and np.array_equal(mean, orc.mean) and np.array_equal(m2, orc.m2)
        assert np.abs(got[0, 1:, 0]).max() > 0  # the wind loads the buildings
        wl.close()


def _lbm_wall(shape, D, steps, precision=1, capacity=256, **kw):
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import LBM, WallLoads
    from tests import helpers as H
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    lbm = LBM(shape, D=D, precision=precision, features=H.FEATURE_SETS["core"], arith=A.ARITH_STRICT, nu=1e-6, f=H.FORCE, omega=H.OMEGA, **H.ZONES)
    lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
    lbm.run(0)
    wl = WallLoads(lbm, capacity=capacity, **kw)
    for _ in range(steps):
        lbm.run(1)
        wl.accumulate()
    out = {"series": wl.series(), "surface": wl.surface(), "summary": wl.summary(), "L": wl.L, "ref": wl.ref_points, "col": wl.column_labels}
    wl.close()
    lbm.close()
    return out, flags


@pytest.mark.gpu
def test_run_to_run_and_host_emulation_and_ring_drains(emu):
    """Two runs give bit-identical series; a capacity of 3 over 7 samples (automatic drains) gives the same series as one drain at the end; the first sample
    == the host-emulated reduction over its per-cell forces."""
    shape = (64, 48, 32)
    a, flags = _lbm_wall(shape, (1, 1, 1), 7)
    b, _ = _lbm_wall(shape, (1, 1, 1), 7, capacity=3)
    assert a["series"].shape == (7, 10, 6) and np.array_equal(a["series"], b["series"])
    one, _ = _lbm_wall(shape, (1, 1, 1), 1)
    assert np.array_equal(one["series"][0], a["series"][0])
    s = one["surface"]
    cells, m, labels, (x, y, z), L, ref = _labelled_list(flags, shape)
    order = np.lexsort((s["cell"], s["label"]))
    F = s["mean_F"][:, order]  # after one sample the mean is the force
    assert np.array_equal(s["cell"][order], cells) and np.array_equal(s["label"][order], labels)
    Px = 64
    dev = (x + (y + z * shape[1]) * Px).astype(np.uint64)
    assert np.array_equal(emu_reduce(emu, shape, Px, dev, F, labels, ref), one["series"][0])
    summ = a["summary"]
    assert summ["samples"] == 7 and np.array_equal(summ["max"], a["series"].max(0)) and np.array_equal(summ["mean"], a["series"].mean(0))


@pytest.mark.gpu
@pytest.mark.parametrize("D", [(2, 1, 1), (1, 2, 1), (1, 1, 2)], ids=["2x1x1", "1x2x1", "1x1x2"])
def test_decompositions_equal_the_single_domain(D):
    """Lists (as global cells), labels, r0 and per-cell statistics bit-identical to the single domain; label loads within 1e-12 relative. In [1,1,2] (Nz = 32:
    blocks of 16 layers) the ground plane lies in the lower block and the roofs reach into the upper one."""
    shape = (64, 48, 32)
    one, flags = _lbm_wall(shape, (1, 1, 1), 5)
    dec, _ = _lbm_wall(shape, D, 5)
    for k in ("cell", "label", "mean_F", "m2_F"):
        assert np.array_equal(one["surface"][k], dec["surface"][k]), k
    assert one["surface"]["samples"] == dec["surface"]["samples"] == 5
    assert np.array_equal(one["ref"], dec["ref"]) and np.array_equal(one["col"], dec["col"]) and one["L"] == dec["L"] == 10
    assert _close(dec["series"], one["series"], floor=1e-14 * np.abs(one["series"]).max())
    cells, _ = W.surface(flags, shape)
    assert np.array_equal(one["surface"]["cell"], cells)
    assert (one["surface"]["z"] >= 16).any()


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
def test_momentum_balance_on_the_device(arith):
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, WallLoads
    shape = (4, 4, 10)
    N = int(np.prod(shape))
    flags = np.zeros((10, 4, 4), np.uint8)
    flags[0] = flags[-1] = TYPE_S
    with Domain(*shape, precision=A.FP32, features=A.VOLUME_FORCE, w=1.0, arith=A.ARITH_STRICT if arith == 0 else A.ARITH_FAST) as d:
        d.rho[:], d.u[:], d.flags[:] = np.ones(N, np.float32), np.zeros(3 * N, np.float32), flags.reshape(-1)
        d.f, d.omega = (1e-5, 0.0, 0.0), (0.0, 0.0, 0.0)
        d.upload_all()
        d.t = 1
        d.enqueue_initialize()
        d.t = 0
        d.run_steps(1920)
        cells = d.solid_surface(3)
        z = cells.astype(np.int64) // 16
        labels = (z > 0).astype(np.uint32)
        wl = WallLoads(d, cells, labels, 2, np.zeros((2, 3)), 3, 4)
        wl.accumulate()
        s = wl.drain()[0]
        F, _, _ = wl.download_cells()
        check_balance(F, z, 10, 1e-5, 128)
        assert abs(s[0, 0] - s[1, 0]) <= 1e-3 * 1.28e-3 and abs(s[0, 0] + s[1, 0] - 1.28e-3) <= 1e-3 * 1.28e-3
        wl.close()


@pytest.mark.gpu
def test_stream_order_ring_full_reset_and_invalid_arguments():
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, WallLoads
    from tests import helpers as H
    shape = (64, 48, 32)
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    Lib = A.lib()
    series = []
    for S in (1, 8):  # drain after every sample / 8 samples back to back, one drain
        with Domain(*shape, precision=A.FP16S, features=H.FEATURE_SETS["luw"], w=cases.relaxation_rate(1e-6), arith=A.ARITH_STRICT, **H.ZONES) as d:
            d.rho[:], d.u[:], d.flags[:] = rho, u, flags
            d.f, d.omega = H.FORCE, H.OMEGA
            d.upload_all()
            d.t = 1
            d.enqueue_initialize()
            d.t = 0
            cells, m, labels, _, L, ref = _labelled_list(flags, shape)
            wl = WallLoads(d, cells, labels, L, ref, 0, S)
            got = []
            for s in range(8):
                d.enqueue_stream_collide()
                d.increment_time_step()
                wl.accumulate()
                if S == 1:
                    got.append(wl.drain())
            if S == 8:
                assert Lib.luw_wall_loads_accumulate(wl._h, d.t) == A.ERR_INVALID  # ring full
                got.append(wl.drain())
                assert wl.drain().shape == (0, L, 6)
                _, _, n = wl.download_cells()
                assert n == 8
                d.finish_queue()
                n0 = d.launch_count()
                wl.accumulate()
                assert d.launch_count() == n0 + 4  # per-cell forces, chunk sums, group sums, label sums
                wl.reset()
                mean, m2, n = wl.download_cells()
                assert n == 0 and not mean.any() and not m2.any() and wl.drain().shape[0] == 0
                # invalid arguments
                h = C.c_void_p()
                c2, l2 = cells[:2].copy(), labels[:2].copy()
                good = dict(cells=c2, labels=l2, L=L, ref=ref, cap=4)

                def create(cells=c2, labels=l2, L=L, ref=ref, cap=4, null_list=False):
                    cells, labels, ref = np.ascontiguousarray(cells, np.uint64), np.ascontiguousarray(labels, np.uint32), np.ascontiguousarray(ref, np.float64)
                    return Lib.luw_wall_loads_create(d._h, cells.size, None if null_list else cells.ctypes.data, labels.ctypes.data, L, ref.ctypes.data, 0, cap,
                                                     C.byref(h))
                assert create(**good) == A.OK
                Lib.luw_wall_loads_destroy(h)
                bad_ref = ref.copy()
                bad_ref[1, 2] = np.inf
                for kw in (dict(cells=c2[::-1].copy(), labels=np.zeros(2, np.uint32)), dict(cells=[c2[0], c2[0]], labels=[0, 0]), dict(cells=[d.N], labels=[0]),
                           dict(labels=[l2[0], L]), dict(L=0), dict(null_list=True), dict(cap=0), dict(ref=bad_ref)):
                    h = C.c_void_p()
                    assert create(**kw) == A.ERR_INVALID and not h.value, kw
            wl.close()
        series.append(np.concatenate(got))
    assert series[0].shape == (8, L, 6) and np.array_equal(series[0], series[1])
    # halo indices are rejected on a decomposed block
    with Domain(34, 24, 16, D=(2, 1, 1), O=(-1, 0, 0), precision=A.FP32, features=0, w=1.0) as d:
        h = C.c_void_p()
        for cell in (0, 33, 1 + 34):
            cl, lb, rf = np.array([cell], np.uint64), np.zeros(1, np.uint32), np.zeros(3)
            rc = Lib.luw_wall_loads_create(d._h, 1, cl.ctypes.data, lb.ctypes.data, 1, rf.ctypes.data, 0, 1, C.byref(h))
            assert rc == (A.OK if cell == 35 else A.ERR_INVALID), cell
            Lib.luw_wall_loads_destroy(h)
            h = C.c_void_p()


@pytest.mark.gpu
def test_cpp_host_layer_equals_the_python_path(tmp_path):
    """LBM_WallLoads (C++ host layer, through luw_host_case's LUW_CASE_WALL_OUT switch) == lbm.WallLoads on the same case, single domain and [1,1,2]."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import LBM, WallLoads
    from tests import helpers as H
    from tests.test_cpp_host import build, run_driver
    build()
    shape, steps, samples = (64, 48, 32), 7, 4
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    feat = H.FEATURE_SETS["core"]
    for D in ((1, 1, 1), (1, 1, 2)):
        path = str(tmp_path / "wall.bin")
        env_keep = dict(os.environ)
        os.environ.update(LUW_CASE_WALL_OUT=path)
        try:
            run_driver(tmp_path, shape, D, 1, feat, 0, 1e-6, steps, flags, rho, u, zones=H.ZONES, stats=samples)
        finally:
            os.environ.clear()
            os.environ.update(env_keep)
        raw = open(path, "rb").read()
        n, L, K = int(np.frombuffer(raw[:8], np.uint64)[0]), int(np.frombuffer(raw[8:12], np.uint32)[0]), int(np.frombuffer(raw[12:20], np.uint64)[0])
        o = 20
        parts = {}
        for key, dt, size in (("series", np.float64, n * L * 6), ("ref", np.float64, 3 * L), ("col", np.uint32, shape[0] * shape[1]), ("cell", np.uint64, K),
                              ("label", np.uint32, K), ("mean_F", np.float32, 3 * K), ("m2_F", np.float32, 3 * K)):
            nb = np.dtype(dt).itemsize * size
            parts[key] = np.frombuffer(raw[o:o + nb], dt)
            o += nb
        assert o == len(raw)
        lbm = LBM(shape, D=D, precision=A.FP16S, features=feat, arith=A.ARITH_STRICT, nu=1e-6, f=H.FORCE, omega=H.OMEGA, **H.ZONES)
        lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
        lbm.run(0)
        wl = WallLoads(lbm)
        lbm.run(steps - samples)
        for _ in range(samples):
            lbm.run(1)
            wl.accumulate()
        py, surf = wl.series(), wl.surface()
        assert n == py.shape[0] == samples and L == wl.L == 10
        assert np.array_equal(parts["series"].reshape(py.shape), py), D
        assert np.array_equal(parts["ref"].reshape(L, 3), wl.ref_points) and np.array_equal(parts["col"].reshape(shape[1], shape[0]), wl.column_labels)
        assert np.array_equal(parts["cell"], surf["cell"]) and np.array_equal(parts["label"], surf["label"])
        assert np.array_equal(parts["mean_F"].reshape(3, K), surf["mean_F"]) and np.array_equal(parts["m2_F"].reshape(3, K), surf["m2_F"])
        wl.close()
        lbm.close()
