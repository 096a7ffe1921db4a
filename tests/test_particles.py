"""Lagrangian tracer particles (csrc/lbm_particles.cuh, luw_particles_*, domain.Particles, lbm.Particles, LBM_Particles) against oracle/particles_oracle.py.
CPU: the Philox block function compiled for the host against numpy's np.random.Philox; the kernel source on host threads against the oracle fed with the
C oracle's update_fields; the ABI surface; lbm.Particles' argument checks. GPU: advance against the oracle on luw_update_fields + a read-back of u, bit for
bit; the lattice is untouched; physics (uniform flow, Poiseuille channel, random-walk moments, walls, open faces, buried releases); bins against
np.histogramdd; ring order and argument errors; stream order; the C++ host layer against Python."""
import ctypes as C
import os
import subprocess
import types

import numpy as np
import pytest

from latticeurbanwind_b200 import cases
from oracle import particles_oracle as PO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UF, VF, EQ, SG, ZONE_BITS, TEMPERATURE = 1, 2, 4, 8, 16 | 32, 64
FEATS = [0, 4, 5, 14, 15]


def _features(feat, thermal=False):
    """The feature sets under test, with nudging and the top sponge on wherever the volume force is (update_fields must ignore them)."""
    return feat | (ZONE_BITS if feat & VF else 0) | (TEMPERATURE if thermal else 0)


def _numpy_philox(ctr, key):
    """The block for counter c is what np.random.Philox gives after one increment from c - 1 (mod 2^256)."""
    c = sum(int(w) << (64 * i) for i, w in enumerate(ctr))
    c = (c - 1) % (1 << 256)
    g = np.random.Philox(counter=np.array([(c >> (64 * i)) & (2 ** 64 - 1) for i in range(4)], np.uint64), key=np.asarray(key, np.uint64))
    return g.random_raw(4)


def _pairs(n=10000, seed=5):
    """(counter, key) pairs: random words, and counters whose low words are 0 / all ones (carries across counter words on numpy's side)."""
    rng = np.random.default_rng(seed)
    ctr = rng.integers(0, 2 ** 64, (n, 4), dtype=np.uint64)
    key = rng.integers(0, 2 ** 64, (n, 2), dtype=np.uint64)
    ctr[: n // 8, 0] = 0
    ctr[n // 8: n // 4, :2] = 0
    ctr[n // 4: n // 4 + 16] = 0
    ctr[n // 4 + 16: n // 4 + 32, :3] = 0
    ctr[n // 4 + 32: n // 4 + 64] = np.uint64(2 ** 64 - 1)
    ctr[:16] = 0
    key[:8] = 0
    ctr[n // 2: n // 2 + 500, 1] = rng.integers(0, 256, 500, dtype=np.uint64)  # the (slot, call, stream, 0) shape the kernels use
    ctr[n // 2: n // 2 + 500, 2:] = 0
    return ctr, key


# ---------------------------------------------------------------------------------------------------------------- CPU: kernel source on host threads
EMU_SRC = r'''
#include "kernels_on_host.cpp"
#include <atomic>
static inline double __dmul_rn(double a, double b) { return a*b; }
static inline double __dadd_rn(double a, double b) { return a+b; }
static inline double __ddiv_rn(double a, double b) { return a/b; }
static inline float __double2float_rn(double a) { return (float)a; }
static inline unsigned atomicAdd(unsigned* a, unsigned v) { return __atomic_fetch_add(a, v, __ATOMIC_RELAXED); }
#include "lbm_particles.cuh"
template<class K> static void launch(unsigned grid, K kernel) {
	emu_blockDim = {256u, 1u, 1u}; emu_gridDim = {grid, 1u, 1u};
	for(unsigned b=0u; b<grid; b++) for(unsigned i=0u; i<256u; i++) { emu_blockIdx = {b, 0u, 0u}; emu_threadIdx = {i, 0u, 0u}; kernel(); }
}
static ParticleSet make_set(double* p, uint8_t* st, uint32_t* em, uint64_t* rel, uint64_t cap, uint64_t seed, uint32_t periodic, uint32_t wall_mode) {
	ParticleSet s; s.p = p; s.state = st; s.emitter = em; s.release = rel; s.capacity = cap; s.seed = seed; s.periodic = periodic; s.wall_mode = wall_mode;
	return s;
}
template<int P, uint32_t F, bool TH> static void run_adv(const DomainConst& c, const StepArgs& a, const ParticleSet& s, uint64_t call, float dt, double sigma, unsigned grid) {
	launch(grid, [&]{ k_particles_advance<P, F, TH>(c, a, s, call, dt, sigma); });
}
template<int P, bool TH> static void pick(const DomainConst& c, const StepArgs& a, const ParticleSet& s, uint64_t call, float dt, double sigma, unsigned grid) {
	if(c.features&F_UPDATE_FIELDS) run_adv<P, F_UPDATE_FIELDS, TH>(c, a, s, call, dt, sigma, grid);
	else switch(c.features&(F_VOLUME_FORCE|F_EQUILIBRIUM)) {
		case 0u: run_adv<P, 0u, TH>(c, a, s, call, dt, sigma, grid); break;
		case F_VOLUME_FORCE: run_adv<P, F_VOLUME_FORCE, TH>(c, a, s, call, dt, sigma, grid); break;
		case F_EQUILIBRIUM: run_adv<P, F_EQUILIBRIUM, TH>(c, a, s, call, dt, sigma, grid); break;
		default: run_adv<P, F_VOLUME_FORCE|F_EQUILIBRIUM, TH>(c, a, s, call, dt, sigma, grid); break;
	}
}
template<int P> static void pick_th(const DomainConst& c, const StepArgs& a, const ParticleSet& s, uint64_t call, float dt, double sigma, unsigned grid) {
	if(c.features&F_TEMPERATURE) pick<P, true>(c, a, s, call, dt, sigma, grid); else pick<P, false>(c, a, s, call, dt, sigma, grid);
}
extern "C" {
void emu_philox(uint64_t n, const uint64_t* ctr, const uint64_t* key, uint64_t* out) { for(uint64_t i=0u; i<n; i++) philox4x64_10(ctr+4u*i, key+2u*i, out+4u*i); }
int emu_particles_advance(const DomainConst* c, const StepArgs* a, double* p, uint8_t* st, uint32_t* em, uint64_t* rel, uint64_t cap, uint64_t seed, uint32_t periodic,
	uint32_t wall_mode, uint64_t call, float dt, double sigma, unsigned grid) {
	const ParticleSet s = make_set(p, st, em, rel, cap, seed, periodic, wall_mode);
	BY_PRECISION(*c, pick_th<P>(*c, *a, s, call, dt, sigma, grid));
	return 0;
}
int emu_particles_emit(const DomainConst* c, double* p, uint8_t* st, uint32_t* em, uint64_t* rel, uint64_t cap, uint64_t seed, uint32_t periodic, const double* box,
	uint32_t per, uint64_t total, uint64_t head, uint64_t call, uint64_t t, unsigned grid) {
	const ParticleSet s = make_set(p, st, em, rel, cap, seed, periodic, 0u);
	launch(grid, [&]{ k_particles_emit(*c, s, box, per, total, head, call, t); });
	return 0;
}
int emu_particles_count(const DomainConst* c, double* p, uint8_t* st, uint64_t cap, const uint32_t* b, const uint32_t* B, uint32_t* bins, unsigned grid) {
	const ParticleSet s = make_set(p, st, nullptr, nullptr, cap, 0u, 0u, 0u);
	launch(grid, [&]{ k_particles_count(*c, s, b[0], b[1], b[2], B[0], B[1], bins); });
	return 0;
}
}
'''


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not os.path.isfile("/usr/local/cuda/include/cuda_fp16.h"):
        pytest.skip("CUDA headers not installed")
    from tests.test_kernel_source_on_host import StepArgs
    d = tmp_path_factory.mktemp("particles_emu")
    src, so = d / "particles_on_host.cpp", str(d / "libparticles_emu.so")
    src.write_text(EMU_SRC)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared", "-fPIC", "-w", "-I/usr/local/cuda/include",
                           "-I" + os.path.join(ROOT, "tests", "host_emulation"), "-I" + os.path.join(ROOT, "latticeurbanwind_b200", "csrc"), str(src), "-o", so])
    L = C.CDLL(so)
    L.emu_sizeof_domain_const.restype = C.c_uint64
    L.emu_make_domain.argtypes = [C.c_void_p] + [C.c_uint32] * 6 + [C.c_int] * 4 + [C.c_uint32, C.c_float, C.c_int, C.c_uint32, C.c_float, C.c_int, C.c_uint32] + \
        [C.c_void_p] * 8 + [C.c_float] * 3
    L.emu_zone_tables.argtypes = [C.c_uint32, C.c_uint32, C.c_float, C.c_void_p, C.c_void_p]
    L.emu_philox.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.emu_particles_advance.argtypes = [C.c_void_p, C.POINTER(StepArgs)] + [C.c_void_p] * 4 + [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_float,
                                                                                                C.c_double, C.c_uint]
    L.emu_particles_emit.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64,
                                                                       C.c_uint64, C.c_uint]
    L.emu_particles_count.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
    return L


def _host_philox(emu, ctr, key):
    ctr, key = np.ascontiguousarray(ctr, np.uint64), np.ascontiguousarray(key, np.uint64)
    out = np.zeros((ctr.shape[0], 4), np.uint64)
    emu.emu_philox(ctr.shape[0], ctr.ctypes.data, key.ctypes.data, out.ctypes.data)
    return out


def test_philox_known_answer_and_numpy(emu):
    """The device Philox function compiled for the host == np.random.Philox: the Random123 known answer and ~10^4 (counter, key) pairs, including counters
    whose low words are 0 (numpy's counter - 1 borrows across words) and all ones. The oracle's vectorised restatement agrees as well."""
    want0 = [0x16554d9eca36314c, 0xdb20fe9d672d0fdc, 0xd7e772cee186176b, 0x7e68b68aec7ba23b]
    assert _host_philox(emu, np.zeros((1, 4)), np.zeros((1, 2)))[0].tolist() == want0
    assert _numpy_philox([0, 0, 0, 0], [0, 0]).tolist() == want0
    ctr, key = _pairs()
    got = _host_philox(emu, ctr, key)
    want = np.stack([_numpy_philox(c, k) for c, k in zip(ctr, key)])
    assert np.array_equal(got, want)
    assert np.array_equal(PO.philox4x64_10(ctr, key), want)


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


# emitters of the (20, 18, 14) case: the ground layer (buildings: BURIED releases), the west and the east face (LEFT with open x faces), the upper middle
CPU_EMITTERS = np.array([[10.0, 9.0, 1.5, 9.5, 8.5, 1.5], [1.0, 9.0, 6.0, 1.0, 3.0, 3.0], [18.5, 4.0, 10.0, 0.5, 3.0, 2.0], [9.3, 8.7, 9.1, 3.2, 2.9, 2.4]])
SUBCASES = [(mask, mode, sigma) for mask in (0, 0b011) for mode in (0, 1) for sigma in (0.0, 0.9)]


class _EmuRing:
    """One particle ring run through the host-compiled kernels, with the same call bookkeeping as luw_particles."""

    def __init__(self, emu, d, capacity, emitters, mask, mode, seed, bins):
        self.emu, self.d, self.cap = emu, d, capacity
        self.p, self.st = np.zeros(3 * capacity), np.zeros(capacity, np.uint8)
        self.em, self.rel = np.zeros(capacity, np.uint32), np.zeros(capacity, np.uint64)
        self.box = np.ascontiguousarray(emitters, np.float64)
        self.mask, self.mode, self.seed = mask, mode, seed
        self.b = np.array(bins, np.uint32)
        self.B = np.array([(n + b - 1) // b for n, b in zip(d.shape, bins)], np.uint32)
        self.bins = np.zeros(int(np.prod(self.B)), np.uint32)
        self.head = self.emit_calls = self.advance_calls = 0

    def _arrays(self):
        return self.p.ctypes.data, self.st.ctypes.data, self.em.ctypes.data, self.rel.ctypes.data

    def emit(self, t, per):
        total = self.box.shape[0] * per
        assert self.emu.emu_particles_emit(self.d.c, *self._arrays(), self.cap, self.seed, self.mask, self.box.ctypes.data, per, total, self.head, self.emit_calls, t, 2) == 0
        self.head = (self.head + total) % self.cap
        self.emit_calls += 1

    def advance(self, args, dt, sigma):
        assert self.emu.emu_particles_advance(self.d.c, C.byref(args), *self._arrays(), self.cap, self.seed, self.mask, self.mode, self.advance_calls, dt, sigma, 1) == 0
        self.advance_calls += 1

    def count(self):
        assert self.emu.emu_particles_count(self.d.c, self.p.ctypes.data, self.st.ctypes.data, self.cap, self.b.ctypes.data, self.B.ctypes.data, self.bins.ctypes.data, 3) == 0


def _same(ring, ref):
    """the device / emulated ring equals the oracle's: positions bit for bit, states, emitters, release times, bins"""
    p = ring["xyz"].T if isinstance(ring, dict) else ring.p.reshape(3, -1)
    st = ring["state"] if isinstance(ring, dict) else ring.st
    assert np.array_equal(p.view(np.uint64), ref.p.view(np.uint64))
    assert np.array_equal(st, ref.state)
    em = ring["emitter"] if isinstance(ring, dict) else ring.em
    rel = ring["release_t"] if isinstance(ring, dict) else ring.rel
    assert np.array_equal(em, ref.emitter) and np.array_equal(rel, ref.release)


@pytest.mark.parametrize("thermal", [False, True], ids=["plain", "thermal"])
@pytest.mark.parametrize("feat", FEATS)
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_kernel_source_equals_the_oracle(emu, precision, feat, thermal):
    """emit, advance and count over several calls at t = 5, 6, 7 (both parities) on the thermal urban case, for periodic masks 0 / 0b011 x wall modes 0 / 1 x
    sigma 0 / 0.9: the host-compiled kernels == the oracle fed with the C oracle's update_fields (the stored u where update_fields leaves it), bit for bit."""
    from oracle import oracle as O
    from tests import helpers as H
    from tests.test_kernel_source_on_host import HostDomain, StepArgs
    shape = H.THERMAL_SHAPE
    N = int(np.prod(shape))
    features = _features(feat, thermal)
    flags, rho0, u0, T0 = _cpu_case(thermal)
    w = cases.relaxation_rate(1e-6)
    orc = O.Oracle().bind(O.make_params(*shape, precision, features, w=w, **H.ZONES))
    fi, gi = np.zeros(19 * N, O.ddf_dtype(precision)), np.zeros(7 * N, O.ddf_dtype(precision))
    rho, u, T = rho0.copy(), u0.copy(), T0.copy()
    if thermal:
        orc.set_thermal(**H.THERMAL)
        orc.initialize_thermal(fi, rho, u, flags, gi, T)
    else:
        orc.initialize(fi, rho, u, flags)
    d = HostDomain(emu, shape, precision, features, w, H.ZONES, thermal=H.THERMAL if thermal else None)
    cap, bins = 300, (3, 4, 5)
    rings = [(_EmuRing(emu, d, cap, CPU_EMITTERS, m, mode, 1000 + k, bins), PO.ParticleRing(shape, cap, CPU_EMITTERS, m, mode, 1000 + k, bins), sigma)
             for k, (m, mode, sigma) in enumerate(SUBCASES)]
    seen = set()
    for t in range(7):
        if thermal:
            orc.stream_collide_thermal(fi, rho, u, flags, t, H.FORCE, H.OMEGA, gi, T)
        else:
            orc.stream_collide(fi, rho, u, flags, t, H.FORCE, H.OMEGA)
        if t < 4:
            continue
        t1 = t + 1
        d.put(d.fi, fi, 19); d.put(d.rho, rho, 1); d.put(d.u, u, 3); d.put(d.flags, flags, 1)
        if thermal:
            d.put(d.gi, gi, 7); d.put(d.T, T, 1)
        r, uu, TT = rho.copy(), u.copy(), T.copy()
        if not feat & UF:
            if thermal:
                orc.update_fields_thermal(fi, r, uu, flags, t1, H.FORCE, H.OMEGA, gi, TT)
            else:
                orc.update_fields(fi, r, uu, flags, t1, H.FORCE, H.OMEGA)
        args = StepArgs(t1, *map(np.float32, H.FORCE), *map(np.float32, H.OMEGA))
        for ring, ref, sigma in rings:
            ring.emit(t1, 25); ref.emit(flags, t1, 25)
            for dt in (6.0, 11.0):
                ring.advance(args, dt, sigma); ref.advance(uu, flags, dt, sigma)
            ring.count(); ref.count()
            _same(ring, ref)
            assert np.array_equal(ring.bins, ref.bins.reshape(-1))
            seen.update(ref.state.tolist())
        assert d.get(d.rho, 1).tobytes() == rho.tobytes() and d.get(d.u, 3).tobytes() == u.tobytes()  # nothing written into the lattice
    assert {PO.ACTIVE, PO.DEPOSITED, PO.LEFT, PO.BURIED} <= seen


# ---------------------------------------------------------------------------------------------------------------- CPU: ABI surface, Python checks
NAMES = ("luw_particles_create", "luw_particles_emit", "luw_particles_advance", "luw_particles_count", "luw_particles_download", "luw_particles_download_bins",
         "luw_particles_reset_bins", "luw_particles_destroy")


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
    em, b, h, n = np.zeros(6), np.ones(3, np.uint32), C.c_void_p(), C.c_uint64(7)
    assert L.luw_particles_create(None, 4, 1, em.ctypes.data, 0, 0, 1, b.ctypes.data, C.byref(h)) == A.ERR_NO_DEVICE and not h.value
    assert L.luw_particles_emit(None, 0, 1) == A.ERR_NO_DEVICE
    assert L.luw_particles_advance(None, 0, *[0.0] * 7, 0.0) == A.ERR_NO_DEVICE
    assert L.luw_particles_count(None) == A.ERR_NO_DEVICE
    assert L.luw_particles_download(None, None, None, None, None) == A.ERR_NO_DEVICE
    assert L.luw_particles_download_bins(None, None, C.byref(n)) == A.ERR_NO_DEVICE and n.value == 7
    assert L.luw_particles_reset_bins(None) == A.ERR_NO_DEVICE
    assert L.luw_particles_destroy(None) == A.ERR_NO_DEVICE
    assert L.luw_last_error_string()


def test_lbm_particles_argument_checks():
    """lbm.Particles rejects a decomposed LBM and every argument luw_particles_create would reject, before it touches a device."""
    from latticeurbanwind_b200.lbm import Particles, particle_args
    lbm = types.SimpleNamespace(D=(2, 1, 1), Ng=(32, 16, 8))
    with pytest.raises(ValueError, match="single domain"):
        Particles(lbm, [[4, 4, 4, 1, 1, 1]], 16)
    Ng = (32, 16, 8)
    good = dict(emitters=[[4, 4, 4, 1, 1, 1]], capacity=16, periodic=(False, False, False), wall_mode=0, bins=(1, 1, 1))
    em, mask, b = particle_args(Ng, **good)
    assert em.shape == (1, 6) and mask == 0 and b.tolist() == [1, 1, 1]
    assert particle_args(Ng, **dict(good, periodic=(True, True, False), emitters=[[-3.0, 40.0, 4, 9, 9, 1]]))[1] == 3  # periodic axes: anywhere
    assert particle_args(Ng, **dict(good, emitters=[[0.5, 0.5, 3.5, 0.5, 0.5, 3.5]]))[0].shape == (1, 6)  # touches 0 and N-1
    for bad in (dict(capacity=0), dict(wall_mode=2), dict(bins=(1, 0, 1)), dict(bins=(1, 1)), dict(periodic=(True, True)),
                dict(emitters=[[4, 4, 4, -1, 1, 1]]), dict(emitters=[[np.nan, 4, 4, 1, 1, 1]]), dict(emitters=[[4, 4, np.inf, 1, 1, 1]]),
                dict(emitters=[[0.5, 4, 4, 1, 1, 1]]), dict(emitters=[[4, 15.5, 4, 1, 1, 1]]), dict(emitters=[[4, 4, 7.5, 1, 1, 0.6]])):
        with pytest.raises(ValueError):
            particle_args(Ng, **dict(good, **bad))
    with pytest.raises(ValueError):
        particle_args((32, 16, 1), **good)  # N < 2 on a non-periodic axis
    assert particle_args((32, 16, 1), **dict(good, periodic=(False, False, True), emitters=[[4, 4, 0, 1, 1, 0]]))[1] == 4


def test_oracle_model_on_hand_made_cases():
    """The oracle's own definitions on cases whose answer is known without it: a uniform field moves by u*dt, interpolation is linear along each axis,
    periodic wrap, LEFT through an open face, the two wall modes, BURIED releases, ring overwrite and bins."""
    shape = (8, 6, 5)
    N = int(np.prod(shape))
    flags = np.zeros(N, np.uint8)
    ring = PO.ParticleRing(shape, 4, [[2.0, 3.0, 2.0, 0.0, 0.0, 0.0]], periodic_mask=0b001, bin_size=(2, 3, 5))
    ring.emit(flags, 3, 2)
    assert ring.state.tolist() == [1, 1, 0, 0] and ring.release.tolist() == [3, 3, 0, 0] and ring.head == 2
    u = np.zeros((3, N), np.float32)
    u[0] = 0.25
    for _ in range(30):
        ring.advance(u, flags, dt=1.0)
    assert np.allclose(ring.p[0, :2], (2.0 + 30 * 0.25) % 8) and (ring.p[0, :2] < 8).all()  # wrapped
    x = np.arange(N) % shape[0]
    u[0] = 0.0
    u[2] = (x * 0.125).astype(np.float32)  # uz linear in x
    ring2 = PO.ParticleRing(shape, 1, [[3.5, 2.0, 2.0, 0.0, 0.0, 0.0]])
    ring2.emit(flags, 0, 1)
    ring2.advance(u, flags, dt=1.0)
    assert ring2.p[:, 0].tolist() == [3.5, 2.0, 2.0 + 3.5 * 0.125]
    ring2.advance(np.full((3, N), 9.0, np.float32), flags, dt=1.0)
    assert ring2.state[0] == PO.LEFT
    flags[3 + (2 + 2 * shape[1]) * shape[0]] = 1  # solid cell (3, 2, 2)
    for mode, want in ((0, PO.ACTIVE), (1, PO.DEPOSITED)):
        r = PO.ParticleRing(shape, 1, [[1.5, 2.0, 2.0, 0.0, 0.0, 0.0]], wall_mode=mode)
        r.emit(flags, 0, 1)
        v = np.zeros((3, N), np.float32)
        v[0] = 1.0
        r.advance(v, flags, dt=1.25)  # 2.75 -> nearest cell 3: solid
        assert r.state[0] == want and r.p[0, 0] == (1.5 if mode == 0 else 2.75)
    r = PO.ParticleRing(shape, 2, [[3.2, 2.0, 2.0, 0.0, 0.0, 0.0], [5.0, 2.0, 2.0, 0.0, 0.0, 0.0]])
    r.emit(flags, 7, 1)
    assert r.state.tolist() == [PO.BURIED, PO.ACTIVE] and r.emitter.tolist() == [0, 1]
    ring.count()
    assert ring.bins.sum() == 2 and ring.samples == 1


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


def _emitters(shape):
    """ground layer, west face, an upper box, and one across the east face"""
    Nx, Ny, Nz = shape
    return np.array([[(Nx - 1) / 2, (Ny - 1) / 2, 1.5, (Nx - 1) / 2, (Ny - 1) / 2, 1.5], [1.0, Ny / 2, Nz / 3, 1.0, Ny / 4, Nz / 5],
                     [Nx / 2 + 0.3, Ny / 3 + 0.1, 2 * Nz / 3, Nx / 5, Ny / 6, Nz / 6], [Nx - 2.0, Ny / 2, Nz / 2, 1.0, Ny / 3, Nz / 4]])


def _snapshot(d):
    """fi, rho, u (and T) bytes of the device lattice"""
    from latticeurbanwind_b200 import _cabi as A
    fi = d.read_fi()
    out = [fi.tobytes()]
    for f, comps in ((A.FIELD_RHO, 1), (A.FIELD_U, 3)) + (((A.FIELD_T, 1),) if d.thermal else ()):
        a = np.empty(comps * d.N, np.float32)
        A.check(A.lib().luw_download(d._h, f, a.ctypes.data, 0, a.size))
        d.finish_queue()
        out.append(a.tobytes())
    return out


def _u_after_update_fields(d, feat):
    """the cell velocities the oracle takes: luw_update_fields + read-back of u (the stored u on UPDATE_FIELDS domains), float32 [3, N]"""
    from latticeurbanwind_b200 import _cabi as A
    if not feat & UF:
        d.enqueue_update_fields()
    u = np.empty(3 * d.N, np.float32)
    A.check(A.lib().luw_download(d._h, A.FIELD_U, u.ctypes.data, 0, u.size))
    d.finish_queue()
    return u.reshape(3, -1)


def _check_rounds(d, flags, feat, pairs, rounds, dt=(7.0, 13.0), per=40, untouched=True):
    """per round: emit, two advances, count on the device and in the oracle (cell velocities from update_fields at the same t), then equal bit for bit.
    pairs: [(domain.Particles, oracle ring, sigma)]"""
    for _ in range(rounds):
        before = _snapshot(d) if untouched else None
        for pt, ref, sigma in pairs:
            pt.emit(per)
            for h in dt:
                pt.advance(h, sigma)
            pt.count()
        if untouched:
            assert _snapshot(d) == before  # emit, advance and count leave fi, rho, u (and T) as they were
        u = _u_after_update_fields(d, feat)
        for pt, ref, sigma in pairs:
            ref.emit(flags, d.t, per)
            for h in dt:
                ref.advance(u, flags, h, sigma)
            ref.count()
            _same(pt.state(), ref)
            b, n = pt.bins()
            assert np.array_equal(b, ref.bins) and n == ref.samples
        d.run_steps(1)


def _pairs_for(d, shape, masks=(0, 0b011), modes=(0, 1), sigmas=(0.0, 0.6), cap=700, bins=(4, 5, 3)):
    from latticeurbanwind_b200.domain import Particles
    em = _emitters(shape)
    out = []
    for k, (m, mode, s) in enumerate((m, mode, s) for m in masks for mode in modes for s in sigmas):
        out.append((Particles(d, em, cap, m, mode, 77 + k, bins), PO.ParticleRing(shape, cap, em, m, mode, 77 + k, bins), s))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("Nx", [63, 64], ids=["padded", "dense"])
@pytest.mark.parametrize("feat", FEATS)
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_advance_equals_the_oracle_on_update_fields(precision, feat, Nx, arith):
    """After 3 steps, two rounds (odd and even t) of emit / advance / count: the device == the oracle fed with luw_update_fields + read-back of u on the same
    domain, bit for bit, for periodic masks 0 / 0b011, both wall modes, sigma 0 and 0.6; the lattice is untouched by the particle calls."""
    shape = (Nx, 48, 32)
    d, flags = _domain(shape, precision, _features(feat), arith)
    with d:
        d.run_steps(3)
        pairs = _pairs_for(d, shape)
        _check_rounds(d, flags, feat, pairs, 2)
        states = set(np.concatenate([ref.state for _, ref, _ in pairs]).tolist())
        assert {PO.ACTIVE, PO.DEPOSITED, PO.LEFT, PO.BURIED} <= states, states
        for pt, _, _ in pairs:
            pt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("feat", [14, 15])
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_thermal_advance_equals_the_oracle(precision, feat, arith):
    """LUW_TEMPERATURE domains (buoyancy enters u through the force): the same bit-identity with update_fields_thermal."""
    shape = (36, 32, 20)
    d, _ = _domain(shape, precision, _features(feat, True), arith, thermal=True)
    flags = np.asarray(d.flags).copy()
    with d:
        d.run_steps(3)
        pairs = _pairs_for(d, shape, masks=(0b011,), sigmas=(0.0, 0.6), cap=500)
        _check_rounds(d, flags, feat, pairs, 2)
        for pt, _, _ in pairs:
            pt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_strict_trajectory_equals_the_c_oracle(precision):
    """50 steps with an advance after each: STRICT device particles == the oracle advected with the C oracle's own flow (stream_collide + update_fields), bit
    for bit, positions and states after every 10 steps."""
    from oracle import oracle as O
    from latticeurbanwind_b200.domain import Particles
    from tests import helpers as H
    shape = (48, 40, 32)
    N = int(np.prod(shape))
    feat = _features(14)
    d, flags = _domain(shape, precision, feat, 0)
    orc = O.Oracle().bind(O.make_params(*shape, precision, feat, w=cases.relaxation_rate(1e-6), **H.ZONES))
    fi = np.zeros(19 * N, O.ddf_dtype(precision))
    _, rho, u = cases.urban(*shape, seed=21, **SMALL)
    rho, u = rho.copy(), u.copy()
    orc.initialize(fi, rho, u, flags)
    em = _emitters(shape)
    with d:
        pt = Particles(d, em, 2000, 0b011, 1, 5, (4, 4, 4))
        ref = PO.ParticleRing(shape, 2000, em, 0b011, 1, 5, (4, 4, 4))
        for s in range(50):
            d.run_steps(1)
            orc.stream_collide(fi, rho, u, flags, s, H.FORCE, H.OMEGA)
            if s % 10 == 0:
                pt.emit(30)
                ref.emit(flags, s + 1, 30)
            pt.advance(4.0, 0.2)
            r, uu = rho.copy(), u.copy()
            orc.update_fields(fi, r, uu, flags, s + 1, H.FORCE, H.OMEGA)
            ref.advance(uu.reshape(3, -1), flags, 4.0, 0.2)
            if s % 10 == 9:
                _same(pt.state(), ref)
        assert (ref.state == PO.ACTIVE).sum() > 100
        pt.close()


def _periodic_domain(shape, u0, features=0, precision=0):
    """fully periodic fluid (no solids, no boundary cells), rho = 1, u = u0 everywhere"""
    from latticeurbanwind_b200.domain import Domain
    d = Domain(*shape, precision=precision, features=features, w=1.0)
    d.rho[:] = 1.0
    N = d.N
    for a in range(3):
        d.u[a * N:(a + 1) * N] = u0[a]
    d.flags[:] = 0
    d.upload_all()
    d.t = 1
    d.enqueue_initialize()
    d.t = 0
    return d


@pytest.mark.gpu
def test_uniform_periodic_flow_moves_particles_by_k_dt_u():
    from latticeurbanwind_b200.domain import Particles
    shape = (32, 24, 16)
    d = _periodic_domain(shape, (0.05, -0.03, 0.02))
    with d:
        d.run_steps(2)
        u = _u_after_update_fields(d, 0)
        uc = u[:, 0].astype(np.float64)
        assert (u == u[:, :1]).all() and np.allclose(uc, (0.05, -0.03, 0.02), rtol=1e-3)  # uniform
        pt = Particles(d, [[15.5, 11.5, 7.5, 15.5, 11.5, 7.5]], 4096, 0b111, 0, 3)
        pt.emit(4096)
        p0 = pt.state()["xyz"]
        k, dt = 80, 7.0  # 28 cells in x: every particle wraps at least once in x
        for _ in range(k):
            pt.advance(dt)
        s = pt.state()
        want = (p0 + k * dt * uc) % np.array(shape, np.float64)
        err = np.abs((s["xyz"] - want + np.array(shape) / 2) % np.array(shape) - np.array(shape) / 2)
        print(f"uniform flow: max |x - (x0 + k dt u) mod N| = {err.max():.3e} cells after {k} advances")
        assert err.max() < 1e-4 and (s["state"] == PO.ACTIVE).all()
        assert ((s["xyz"] >= 0) & (s["xyz"] < np.array(shape))).all()
        pt.close()


@pytest.mark.gpu
def test_poiseuille_channel_displacement_matches_the_interpolated_parabola():
    """Force-driven channel between solid layers z = 0 and z = Nz-1 (walls half way to the fluid), periodic x / y, sigma = 0: one advance moves each particle
    in x by dt times the parabola u(z) = f/(2 nu) (z - 1/2)(Nz - 3/2 - z) interpolated between its two z cells. Tolerance: dt times the largest deviation of the
    lattice's own cell velocities from the parabola (the interpolation weights sum to one), plus float rounding. No particle enters a wall."""
    from latticeurbanwind_b200.domain import Domain, Particles
    shape = (32, 8, 18)
    Nx, Ny, Nz = shape
    f, nu = 1e-5, 1.0 / 6.0
    d = Domain(*shape, precision=0, features=VF, w=1.0)
    z = np.arange(d.N) // (Nx * Ny)
    d.flags[:] = np.where((z == 0) | (z == Nz - 1), 1, 0).astype(np.uint8)
    d.rho[:] = 1.0
    d.upload_all()
    d.f = (f, 0.0, 0.0)
    d.t = 1
    d.enqueue_initialize()
    d.t = 0
    with d:
        d.run_steps(6000)
        u = _u_after_update_fields(d, VF)
        zc = np.arange(Nz, dtype=np.float64)
        par = np.where((zc >= 1) & (zc <= Nz - 2), f / (2 * nu) * (zc - 0.5) * (Nz - 1.5 - zc), 0.0)
        fluid = (z >= 1) & (z <= Nz - 2)
        lattice_err = np.abs(u[0][fluid] - par[z[fluid]]).max()
        umax = par.max()
        pt = Particles(d, [[(Nx - 1) / 2, (Ny - 1) / 2, (Nz - 1) / 2, (Nx - 1) / 2, (Ny - 1) / 2, (Nz - 3) / 2]], 20000, 0b011, 0, 9)
        pt.emit(20000)
        s0 = pt.state()
        dt = 10.0
        pt.advance(dt)
        s1 = pt.state()
        pz = s0["xyz"][:, 2]
        z0 = np.minimum(np.floor(pz).astype(np.int64), Nz - 2)
        fz = pz - z0
        want = dt * (par[z0] * (1 - fz) + par[z0 + 1] * fz)
        dx = (s1["xyz"][:, 0] - s0["xyz"][:, 0] + Nx / 2) % Nx - Nx / 2
        err = np.abs(dx - want).max()
        tol = dt * (lattice_err + 1e-6 * umax)
        print(f"Poiseuille: umax = {umax:.4e}, lattice max |u - parabola| = {lattice_err:.3e} ({lattice_err / umax:.2%} of umax), "
              f"particle max |dx - dt u_interp| = {err:.3e}, tolerance {tol:.3e}")
        assert lattice_err < 0.05 * umax and err <= tol
        assert (s1["state"] == PO.ACTIVE).all()
        assert (np.abs(s1["xyz"][:, 2] - pz) < 1e-6 * dt).all()
        nz = np.floor(s1["xyz"][:, 2] + 0.5)
        assert ((nz >= 1) & (nz <= Nz - 2)).all()  # no particle in a wall cell
        pt.close()


@pytest.mark.gpu
def test_random_walk_moments_in_quiescent_fluid():
    """2^20 particles, n = 4 advances with sigma = 0.7 in fluid at rest: per axis the mean displacement is within 5 standard errors of 0 and the mean squared
    displacement within 5 standard errors of n sigma^2 (a sum of n uniform steps: Var(d^2) = sigma^4 (2 n^2 - 6 n / 5))."""
    from latticeurbanwind_b200.domain import Particles
    shape = (64, 64, 64)
    d = _periodic_domain(shape, (0.0, 0.0, 0.0))
    M, n, sigma = 1 << 20, 4, 0.7
    with d:
        d.run_steps(1)
        assert not _u_after_update_fields(d, 0).any()
        pt = Particles(d, [[31.5, 31.5, 31.5, 31.5, 31.5, 31.5]], M, 0b111, 0, 12345)
        pt.emit(M)
        p0 = pt.state()["xyz"]
        for _ in range(n):
            pt.advance(1.0, sigma)
        disp = (pt.state()["xyz"] - p0 + 32.0) % 64.0 - 32.0
        se_mean = np.sqrt(n * sigma ** 2 / M)
        se_msd = np.sqrt(sigma ** 4 * (2 * n * n - 1.2 * n) / M)
        mean, msd = disp.mean(axis=0), (disp ** 2).mean(axis=0)
        print(f"random walk: mean {mean} (5 se = {5 * se_mean:.2e}), msd {msd} against {n * sigma ** 2} (5 se = {5 * se_msd:.2e})")
        assert (np.abs(mean) < 5 * se_mean).all() and (np.abs(msd - n * sigma ** 2) < 5 * se_msd).all()
        pt.close()


def _solid(flags, shape, q):
    Nx, Ny, Nz = shape
    n = [np.floor(q[:, a] + 0.5).astype(np.int64) % shape[a] for a in range(3)]
    return (flags[n[0] + (n[1] + n[2] * Ny) * Nx] & 3) == 1, n


@pytest.mark.gpu
def test_walls_open_faces_and_buried_releases():
    """Urban case, sigma > 0. Mode 0: every ACTIVE particle sits in a non-solid cell, none is DEPOSITED, and ACTIVE + LEFT is conserved. Mode 1: every
    DEPOSITED particle's cell is TYPE_S and has a non-solid cell among its 26 neighbours. Open faces produce LEFT particles, which never move again;
    releases into solid cells are BURIED and never move."""
    from latticeurbanwind_b200.domain import Particles
    shape = (64, 48, 32)
    d, flags = _domain(shape, 1, _features(14), 1)
    em = _emitters(shape)
    with d:
        d.run_steps(3)
        for mode in (0, 1):
            pt = Particles(d, em, 4000, 0, mode, 31)
            pt.emit(1000)
            s0 = pt.state()
            live0 = (s0["state"] == PO.ACTIVE).sum()
            buried0 = s0["state"] == PO.BURIED
            assert buried0.any() and _solid(flags, shape, s0["xyz"][buried0])[0].all()
            assert not _solid(flags, shape, s0["xyz"][s0["state"] == PO.ACTIVE])[0].any()
            left_at = None
            for k in range(30):  # |u| dt + sigma sqrt(3) < 1 cell per axis: a deposit lands next to the cell the particle came from
                pt.advance(1.5, 0.35)
                if k == 14:
                    left_at = pt.state()
            s = pt.state()
            st = s["state"]
            active = st == PO.ACTIVE
            assert not _solid(flags, shape, s["xyz"][active])[0].any()
            assert (st == PO.LEFT).any()
            out = (s["xyz"] < 0) | (s["xyz"] > np.array(shape) - 1)
            assert out[st == PO.LEFT].any(axis=1).all() and not out[active].any()
            was_left = left_at["state"] == PO.LEFT
            assert np.array_equal(s["xyz"][was_left], left_at["xyz"][was_left])  # LEFT particles stay where they left
            assert np.array_equal(s["xyz"][buried0], s0["xyz"][buried0]) and (st[buried0] == PO.BURIED).all()
            if mode == 0:
                assert not (st == PO.DEPOSITED).any() and active.sum() + (st == PO.LEFT).sum() == live0
            else:
                dep = st == PO.DEPOSITED
                assert dep.any()
                solid, n = _solid(flags, shape, s["xyz"][dep])
                assert solid.all()
                Nx, Ny, Nz = shape
                touches = np.zeros(dep.sum(), bool)
                for dx in (-1, 0, 1):
                    for dy in (-1, 0, 1):
                        for dz in (-1, 0, 1):
                            x, y, z = n[0] + dx, n[1] + dy, n[2] + dz
                            ok = (x >= 0) & (x < Nx) & (y >= 0) & (y < Ny) & (z >= 0) & (z < Nz)
                            idx = np.clip(x, 0, Nx - 1) + (np.clip(y, 0, Ny - 1) + np.clip(z, 0, Nz - 1) * Ny) * Nx
                            touches |= ok & ((flags[idx] & 3) != 1)
                assert touches.all()
            pt.close()


@pytest.mark.gpu
def test_bins_equal_histogramdd_and_reset():
    from latticeurbanwind_b200.domain import Particles
    shape = (64, 48, 32)
    d, flags = _domain(shape, 0, _features(14), 1)
    bins = (5, 7, 3)
    edges = [np.arange(0, -(-n // b) + 1) for n, b in zip(shape, bins)]
    with d:
        d.run_steps(2)
        pt = Particles(d, _emitters(shape), 3000, 0b011, 0, 8, bins)
        want = np.zeros([len(e) - 1 for e in edges], np.int64)
        for k in range(6):
            pt.emit(200)
            pt.advance(5.0, 0.5)
            pt.count()
            s = pt.state()
            a = s["xyz"][s["state"] == PO.ACTIVE]
            cell = np.floor(a + 0.5).astype(np.int64) % np.array(shape)
            h, _ = np.histogramdd(cell // np.array(bins), bins=edges)
            want += h.astype(np.int64)
            d.run_steps(1)
        got, n = pt.bins()
        assert n == 6 and got.shape == tuple(len(e) - 1 for e in edges[::-1])
        assert np.array_equal(got.astype(np.int64), want.transpose(2, 1, 0)) and want.sum() > 1000
        pt.reset_bins()
        got, n = pt.bins()
        assert n == 0 and not got.any()
        pt.close()


@pytest.mark.gpu
def test_ring_order_release_times_and_invalid_arguments():
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, Particles
    Lib = A.lib()
    shape = (32, 24, 16)
    d = _periodic_domain(shape, (0.0, 0.0, 0.0))
    with d:
        em = [[5.0, 5.0, 5.0, 1.0, 1.0, 1.0], [20.0, 12.0, 9.0, 2.0, 2.0, 2.0]]
        pt = Particles(d, em, 10, 0, 0, 1)
        assert (pt.state()["state"] == PO.FREE).all()
        n0 = d.launch_count()
        for t in (5, 6, 7):
            pt.emit(3, t=t)
        assert d.launch_count() == n0 + 3  # one kernel per call
        s = pt.state()
        # slots 0-5 at t = 5, 6-9 and 0-1 at t = 6, 2-7 at t = 7: order [emitter][i], the oldest overwritten
        assert s["release_t"].tolist() == [6, 6, 7, 7, 7, 7, 7, 7, 6, 6]
        assert s["emitter"].tolist() == [1, 1, 0, 0, 0, 1, 1, 1, 0, 1]
        assert (s["state"] == PO.ACTIVE).all()
        box = np.array(em)[s["emitter"]]
        assert (np.abs(s["xyz"] - box[:, :3]) <= box[:, 3:]).all()
        ref = PO.ParticleRing(shape, 10, em, 0, 0, 1)
        for t in (5, 6, 7):
            ref.emit(np.zeros(d.N, np.uint8), t, 3)
        _same(s, ref)
        pt.emit(0)
        assert np.array_equal(pt.state()["release_t"], s["release_t"])
        h = C.c_void_p()
        assert Lib.luw_particles_emit(pt._h, 0, 6) == A.ERR_INVALID  # 2 * 6 > 10
        for bad in (float("nan"), float("inf"), -0.5):
            assert Lib.luw_particles_advance(pt._h, d.t, *[0.0] * 6, 1.0, bad) == A.ERR_INVALID
        assert Lib.luw_particles_advance(pt._h, d.t, *[0.0] * 6, float("inf"), 0.0) == A.ERR_INVALID
        pt.close()

        def create(em=em, cap=8, mask=0, mode=0, b=(1, 1, 1), dom=None, null=()):
            e = np.ascontiguousarray(em, np.float64)
            bb = np.ascontiguousarray(b, np.uint32)
            h = C.c_void_p()
            rc = Lib.luw_particles_create(None if "dom" in null else (dom or d)._h, cap, e.size // 6, None if "em" in null else e.ctypes.data, mask, mode, 1,
                                          None if "bins" in null else bb.ctypes.data, None if "out" in null else C.byref(h))
            if rc == A.OK:
                Lib.luw_particles_destroy(h)
            else:
                assert not h.value
            return rc
        assert create() == A.OK and create(em=np.zeros((0, 6))) == A.OK
        assert create(em=[[-3.0, 30.0, 5.0, 9.0, 9.0, 1.0]], mask=0b011) == A.OK  # periodic axes: anywhere
        for kw in (dict(cap=0), dict(mode=2), dict(b=(1, 0, 1)), dict(em=[[0.5, 5, 5, 1, 1, 1]]), dict(em=[[5, 5, 15.5, 1, 1, 1]]),
                   dict(em=[[5, 5, 5, -1, 1, 1]]), dict(em=[[np.nan, 5, 5, 1, 1, 1]]), dict(em=[[5, 5, 5, 1, np.inf, 1]]),
                   dict(null=("dom",)), dict(null=("em",)), dict(null=("bins",)), dict(null=("out",))):
            assert create(**kw) == A.ERR_INVALID, kw
    with Domain(34, 24, 16, D=(2, 1, 1), O=(-1, 0, 0), precision=A.FP32, features=0, w=1.0) as dec:  # a decomposed block
        assert create(dom=dec) == A.ERR_INVALID
    with Domain(16, 16, 1, precision=A.FP32, features=0, w=1.0) as flat:  # N < 2 on a non-periodic axis
        assert create(dom=flat, em=[[5, 5, 0, 1, 1, 0]]) == A.ERR_INVALID
        assert create(dom=flat, em=[[5, 5, 0, 1, 1, 0]], mask=0b100) == A.OK


@pytest.mark.gpu
def test_stream_order_without_synchronisation():
    """200 steps with an advance (and every 10th an emit and a count) after each, no host synchronisation in between == the same run synchronised after
    every call."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Particles
    shape = (64, 48, 32)
    feat = _features(14)
    res = []
    for sync in (False, True):
        d, _ = _domain(shape, A.FP16S, feat, 1)
        with d:
            pt = Particles(d, _emitters(shape), 5000, 0b011, 1, 4, (8, 8, 8))
            for s in range(200):
                d.run_steps(1)
                if s % 10 == 0:
                    pt.emit(100)
                    if sync:
                        d.finish_queue()
                pt.advance(2.0, 0.3)
                if sync:
                    d.finish_queue()
                if s % 10 == 9:
                    pt.count()
            res.append((pt.state(), pt.bins()))
            pt.close()
    (a, ba), (b, bb) = res
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(ba[0], bb[0]) and ba[1] == bb[1] == 20
    assert (a["state"] == PO.ACTIVE).sum() > 500


@pytest.mark.gpu
def test_cpp_host_layer_equals_the_python_path(tmp_path):
    """LBM_Particles (C++ host layer, through luw_host_case's LUW_CASE_PARTICLES switch) == lbm.Particles on the same case, bit for bit."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import LBM, Particles
    from tests import helpers as H
    from tests.test_cpp_host import build, run_driver
    build()
    shape, steps, samples = (64, 48, 32), 9, 6
    flags, rho, u = cases.urban(*shape, seed=21, **SMALL)
    feat = _features(14)
    em = _emitters(shape)
    cap, per, mask, mode, seed, bins, dt, sigma = 3000, 50, 0b011, 1, 17, (4, 6, 8), 3.0, 0.4
    path = str(tmp_path / "particles.bin")
    env_keep = dict(os.environ)
    os.environ.update(LUW_CASE_PARTICLES=",".join(repr(float(v)) for v in em.reshape(-1)), LUW_CASE_PARTICLES_OUT=path,
                      LUW_CASE_PARTICLES_ARGS=",".join(str(v) for v in (cap, per, mask, mode, seed, *bins, dt, sigma)))
    try:
        run_driver(tmp_path, shape, (1, 1, 1), A.FP16S, feat, 0, 1e-6, steps, flags, rho, u, zones=H.ZONES, stats=samples)
    finally:
        os.environ.clear()
        os.environ.update(env_keep)
    raw = open(path, "rb").read()
    K = int(np.frombuffer(raw[:8], np.uint64)[0])
    o = 8
    xyz = np.frombuffer(raw[o:o + 24 * K], np.float64).reshape(3, K); o += 24 * K
    st = np.frombuffer(raw[o:o + K], np.uint8); o += K
    emi = np.frombuffer(raw[o:o + 4 * K], np.uint32); o += 4 * K
    rel = np.frombuffer(raw[o:o + 8 * K], np.uint64); o += 8 * K
    n = int(np.frombuffer(raw[o:o + 8], np.uint64)[0]); o += 8
    cbins = np.frombuffer(raw[o:], np.uint32)
    lbm = LBM(shape, precision=A.FP16S, features=feat, arith=A.ARITH_STRICT, nu=1e-6, f=H.FORCE, omega=H.OMEGA, **H.ZONES)
    lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
    lbm.run(0)
    lbm.run(steps - samples)
    pt = Particles(lbm, em, cap, (True, True, False), mode, seed, bins)
    for _ in range(samples):
        lbm.run(1)
        pt.emit(per)
        pt.advance(dt, sigma)
        pt.count()
    s = pt.state()
    b, nb = pt.bins()
    assert K == cap and n == nb == samples
    assert np.array_equal(xyz.T.view(np.uint64), s["xyz"].view(np.uint64)) and np.array_equal(st, s["state"])
    assert np.array_equal(emi, s["emitter"]) and np.array_equal(rel, s["release_t"]) and np.array_equal(cbins, b.reshape(-1))
    assert (s["state"] == PO.ACTIVE).sum() > 100
    pt.close()
    lbm.close()

