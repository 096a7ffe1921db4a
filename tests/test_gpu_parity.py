"""GPU parity: CUDA path through the C ABI vs the CPU oracle on identical seeded inputs.

Bars (BASELINE.json north_star): flags and cell indexing bit-exact; u / rho within a stated tolerance after N steps.
 * LUW_ARITH_STRICT: the kernels evaluate the reference's expressions as written -> every DDF, rho and u value must be EQUAL to the
   oracle's (the oracle itself is pinned bit-for-bit to the reference kernel text, tests/test_oracle_vs_reference.py).
 * LUW_ARITH_FAST: contraction allowed -> tolerance stated below.
"""
import numpy as np
import pytest

from latticeurbanwind_b200 import cases
from tests import helpers as H

pytestmark = pytest.mark.gpu

STEPS = 24
# FAST-mode tolerances after STEPS steps on the small urban case (lattice units; c_s = 0.577, |u| <= 0.17)
TOL_FAST = {0: dict(rel_l2_u=2e-5, max_abs_u=2e-6, rel_l2_rho=1e-6), 1: dict(rel_l2_u=2e-3, max_abs_u=4e-4, rel_l2_rho=1e-4), 2: dict(rel_l2_u=1e-3, max_abs_u=2e-4, rel_l2_rho=1e-4)}


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("fset", ["bench", "plain", "core", "luw", "luwnf"])
def test_strict_equals_oracle(oracle_lib, precision, fset):
    O = oracle_lib
    shape = (48, 40, 32)
    flags, rho, u = H.small_urban(*shape)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS[fset]
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, STEPS, w)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, STEPS, w, arith=0)
    assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision)), "DDFs differ"
    assert np.array_equal(got[1], ref[1]), "rho differs"
    assert np.array_equal(got[2], ref[2]), "u differs"


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_fast_within_tolerance(oracle_lib, precision):
    O = oracle_lib
    shape = (48, 40, 32)
    flags, rho, u = H.small_urban(*shape)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS["luw"]
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, STEPS, w)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, STEPS, w, arith=1)
    tol = TOL_FAST[precision]
    e = H.errors(got, ref)
    H.report("fast_within_tolerance", precision=precision, steps=STEPS, rel_l2_u=e[0], max_abs_u=e[1], rel_l2_rho=e[2], tol=tol)
    assert H.rel_l2(got[2], ref[2]) <= tol["rel_l2_u"]
    assert float(np.abs(got[2] - ref[2]).max()) <= tol["max_abs_u"]
    assert H.rel_l2(got[1], ref[1]) <= tol["rel_l2_rho"]


def test_update_fields_on_demand(oracle_lib):
    """Without UPDATE_FIELDS the host sees rho/u only after update_fields (FX/lbm.hpp:406-412)."""
    O = oracle_lib
    shape = (32, 24, 16)
    flags, rho, u = H.small_urban(*shape)
    w = cases.relaxation_rate(1e-4)
    feat = H.FEATURE_SETS["luwnf"]
    for precision in (0, 1):
        ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, 7, w, update_at_end=True)
        got = H.run_cuda(shape, precision, feat, flags, rho, u, 7, w, arith=0, update_at_end=True, batched=True)
        assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])


# ---------------------------------------------------------------------------------------------- the TMA-tiled step kernel
TILED_SHAPES = [(64, 8, 4), (128, 20, 12), (80, 10, 7), (192, 9, 5), (768, 6, 4), (66, 10, 6), (130, 7, 5), (202, 6, 4), (65, 8, 4), (129, 7, 5), (253, 10, 7), (385, 5, 3)]  # the last four: odd Nx (the row's last pair holds one cell; real decks size Nx = round(si_x / cell), FX/setup.cpp:3552-3568); exact tiles, several tiles, partial tiles in x / y / z, strips longer than the stage ring, x extents that need a padded device row pitch (decomposed blocks: Nx/Dx + 2)


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("fset", ["bench", "plain", "luw", "luwnf"])
@pytest.mark.parametrize("shape", TILED_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_tiled_strict_equals_oracle(oracle_lib, precision, fset, shape):
    O = oracle_lib
    flags, rho, u = cases.urban(*shape, seed=77, edge=3, pitch=6)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS[fset]
    zones = dict(downstream_face=2, buffer_N=3, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=2, sponge_inv_tau=0.02)
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, 9, w, zones=zones)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, 9, w, arith=0, zones=zones, expect_tiles=True)
    assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision)), "DDFs differ"
    assert np.array_equal(got[1], ref[1]), "rho differs"
    assert np.array_equal(got[2], ref[2]), "u differs"


@pytest.mark.parametrize("odd", [False, True], ids=["even", "oddNx"])
@pytest.mark.parametrize("precision", [0, 1], ids=["fp32", "fp16s"])
def test_tiled_periodic_box_equals_oracle(oracle_lib, precision, odd):
    """Fully periodic lattice (upstream BENCHMARK protocol): every wrapped neighbour goes through the tile kernel's boundary patch. Odd Nx: the periodic-x
    neighbour of the last column belongs to cell 0 of the row's last pair."""
    O = oracle_lib
    shape = (128, 12, 6) if precision == 0 else (768, 6, 4)  # one tile per strip / strips longer than the stage ring (parked column without the barrier)
    if odd:
        shape = (127, 12, 6) if precision == 0 else (771, 6, 4)  # wrap inside the only tile / through the parked column
    flags, rho, u = cases.periodic_box(*shape, seed=5, amp=1e-2)
    w = cases.relaxation_rate(1.0 / 6.0)
    ref = H.run_cpu(O.Oracle(), O, shape, precision, 0, flags, rho, u, 11, w)
    got = H.run_cuda(shape, precision, 0, flags, rho, u, 11, w, arith=0, expect_tiles=True)
    assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision))


@pytest.mark.parametrize("precision", [0, 1], ids=["fp32", "fp16s"])
def test_tiled_decomposed_block_equals_oracle(oracle_lib, precision):
    """One block of a 2x2x2 decomposition: halo cells must not execute, their slots must survive the tile write-back unchanged."""
    O = oracle_lib
    glob = (124, 20, 12)
    flags, rho, u = cases.urban(*glob, seed=3, edge=3, pitch=6)
    shape, Ov, flags, rho, u = H.cut_block(glob, (2, 2, 2), (1, 0, 1), flags, rho, u)
    assert shape == (64, 12, 8)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS["luw"]
    zones = dict(downstream_face=2, buffer_N=3, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=2, sponge_inv_tau=0.02)
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, 5, w, zones=zones, D=(2, 2, 2), Ov=Ov)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, 5, w, arith=0, zones=zones, D=(2, 2, 2), O=Ov, expect_tiles=True)
    assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision))
    assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])


TOL_TILED_FAST = {0: dict(rel_l2_u=2e-5, max_abs_u=3e-6, rel_l2_rho=1e-6), 1: dict(rel_l2_u=2e-3, max_abs_u=4e-4, rel_l2_rho=1e-4), 2: dict(rel_l2_u=1e-3, max_abs_u=2e-4, rel_l2_rho=1e-4)}


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("fset", ["bench", "luw"])
def test_tiled_fast_within_tolerance(oracle_lib, precision, fset):
    O = oracle_lib
    shape = (128, 40, 24)
    flags, rho, u = cases.urban(*shape, seed=11, edge=6, pitch=12)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS[fset]
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, STEPS, w, update_at_end=(fset == "bench"))
    got = H.run_cuda(shape, precision, feat, flags, rho, u, STEPS, w, arith=1, update_at_end=(fset == "bench"), expect_tiles=True)
    tol = TOL_TILED_FAST[precision]
    e = H.errors(got, ref)
    H.report("tiled_fast_within_tolerance", precision=precision, fset=fset, steps=STEPS, rel_l2_u=e[0], max_abs_u=e[1], rel_l2_rho=e[2], tol=tol)
    assert H.rel_l2(got[2], ref[2]) <= tol["rel_l2_u"]
    assert float(np.abs(got[2] - ref[2]).max()) <= tol["max_abs_u"]
    assert H.rel_l2(got[1], ref[1]) <= tol["rel_l2_rho"]


# ---------------------------------------------------------------------------------------------- the instantiations bench.py times
# bench.py's workloads: "chan" (FEAT = 4, channel case: TYPE_E x faces, TYPE_S walls) and "luwnf" / "luw" (FEAT = 14 / 15, urban case), FAST arithmetic, the tile
# variant the dispatcher picks (csrc/lbm_launch.inc choose_tile). Every variant the dispatcher can pick is pinned here, STRICT bit for bit and FAST within tolerance.
BENCH_CASES = {"chan": ("channel", 1.0 / 6.0), "luwnf": ("urban", 1e-6), "luw": ("urban", 1e-6)}
BENCH_VARIANTS = [0, 1, 3, 4, 5]  # V0 / V1 two-pass 128x2, V3 single-pass, V4 two-pass 128x4, V5 the lean-loop kernel (default for FAST two-pass configurations)
BENCH_ZONES = dict(downstream_face=2, buffer_N=5, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=4, sponge_inv_tau=0.02)


def _bench_case(fset, shape):
    case, nu = BENCH_CASES[fset]
    flags, rho, u = cases.block_case(case, shape, edge=4, pitch=8)
    return flags, rho, u, cases.relaxation_rate(nu)


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("variant", BENCH_VARIANTS, ids=lambda v: f"V{v}")
@pytest.mark.parametrize("fset", ["chan", "luwnf", "luw"])
def test_bench_instantiation_strict_equals_oracle(oracle_lib, monkeypatch, precision, variant, fset):
    O = oracle_lib
    shape = (256, 24, 12)
    flags, rho, u, w = _bench_case(fset, shape)
    feat = H.FEATURE_SETS[fset]
    uae = not (feat & 1)
    monkeypatch.setenv("LUW_TILE_VARIANT", str(variant))
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, 9, w, zones=BENCH_ZONES, update_at_end=uae)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, 9, w, arith=0, zones=BENCH_ZONES, update_at_end=uae, expect_tiles=True)
    assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision)), "DDFs differ"
    assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2]), "rho / u differ"


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("variant", BENCH_VARIANTS, ids=lambda v: f"V{v}")
@pytest.mark.parametrize("fset", ["chan", "luwnf", "luw"])
def test_bench_instantiation_fast_within_tolerance(oracle_lib, monkeypatch, precision, variant, fset):
    O = oracle_lib
    shape = (256, 24, 12)
    flags, rho, u, w = _bench_case(fset, shape)
    feat = H.FEATURE_SETS[fset]
    uae = not (feat & 1)
    monkeypatch.setenv("LUW_TILE_VARIANT", str(variant))
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, STEPS, w, zones=BENCH_ZONES, update_at_end=uae)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, STEPS, w, arith=1, zones=BENCH_ZONES, update_at_end=uae, expect_tiles=True)
    tol = TOL_TILED_FAST[precision]
    e = H.errors(got, ref)
    H.report("bench_instantiation_fast", precision=precision, variant=variant, fset=fset, steps=STEPS, rel_l2_u=e[0], max_abs_u=e[1], rel_l2_rho=e[2], tol=tol)
    assert e[0] <= tol["rel_l2_u"] and e[1] <= tol["max_abs_u"] and e[2] <= tol["rel_l2_rho"], e


@pytest.mark.parametrize("shape", [(256, 24, 12), (253, 12, 9)], ids=["256x24x12", "253x12x9-oddNx"])
@pytest.mark.parametrize("variant", [0, 4, 5, 6, 7], ids=lambda v: f"V{v}")
def test_fast_result_does_not_depend_on_the_tile_variant(monkeypatch, variant, shape):
    """A cell's FAST result is a function of its own DDFs only (DESIGN.md 3.1): every two-pass variant -- tile shape, lean or general loop, masked or
    unmasked stores -- must produce the same bits. This is what makes decomposed FAST runs equal to single-domain ones."""
    flags, rho, u, w = _bench_case("luw", shape)
    res = []
    for v in (1, variant):
        monkeypatch.setenv("LUW_TILE_VARIANT", str(v))
        res.append(H.run_cuda(shape, 1, H.FEATURE_SETS["luw"], flags, rho, u, 11, w, arith=1, zones=BENCH_ZONES, expect_tiles=True))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][2], res[1][2])


@pytest.mark.parametrize("variant,shape", [(5, (256, 24, 12)), (7, (256, 24, 12))], ids=["V5-lean", "V7-64wide"])
def test_fp32_two_pass_variants_agree(monkeypatch, variant, shape):
    """The FP32 LES step runs two-pass by default (V1; the lean loop V5 on large lattices; V7 = two-pass on 64-wide tiles for blocks narrower than 128 cells,
    csrc/lbm_launch.inc choose_tile): all three must produce V1's bits, or a decomposed FP32 run would depend on how wide its blocks are."""
    flags, rho, u, w = _bench_case("luw", shape)
    res = []
    for v in (1, variant):
        monkeypatch.setenv("LUW_TILE_VARIANT", str(v))
        res.append(H.run_cuda(shape, 0, H.FEATURE_SETS["luw"], flags, rho, u, 11, w, arith=1, zones=BENCH_ZONES, expect_tiles=True))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][2], res[1][2])


@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
def test_fp32_les_on_a_narrow_lattice_takes_the_64_wide_two_pass_tiles(oracle_lib, monkeypatch, arith):
    """66 cells wide (a block of a 128-cell lattice split in x): no explicit variant, so choose_tile falls through V1 to V7. STRICT equals the oracle bit for bit, FAST within tolerance."""
    O = oracle_lib
    monkeypatch.delenv("LUW_TILE_VARIANT", raising=False)
    shape = (66, 24, 12)
    flags, rho, u, w = _bench_case("luw", shape)
    feat = H.FEATURE_SETS["luw"]
    ref = H.run_cpu(O.Oracle(), O, shape, 0, feat, flags, rho, u, 9, w, zones=BENCH_ZONES)
    got = H.run_cuda(shape, 0, feat, flags, rho, u, 9, w, arith=arith, zones=BENCH_ZONES, expect_tiles=True)
    if arith == 0:
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
    else:
        e = H.errors(got, ref)
        tol = TOL_TILED_FAST[0]
        assert e[0] <= tol["rel_l2_u"] and e[1] <= tol["max_abs_u"] and e[2] <= tol["rel_l2_rho"], e


# 100 steps at BASELINE configs[0] size (SURVEY 8c: "FP16S: CUDA-FP16S vs oracle-FP16S, rel-L2(u) <= 1e-4 after 100 steps" was a proposal to be calibrated).
# Measured values are printed and recorded (gpurun_out/parity_measured.jsonl -> profiles/); the bars are <= 3x measured. For the 16-bit formats the floor
# is the storage format itself: a FAST value that differs from the STRICT one in its last float bits rounds to the neighbouring 16-bit code with
# probability ~1e-4 per DDF and step, and one code is 2^-11 of a DDF -- that, not the arithmetic, is what separates two FP16 trajectories.
TOL_C1_100 = {0: dict(rel_l2_u=3e-5, max_abs_u=5e-6, rel_l2_rho=3e-6), 1: dict(rel_l2_u=2e-3, max_abs_u=1e-3, rel_l2_rho=2e-4), 2: dict(rel_l2_u=2e-3, max_abs_u=1e-3, rel_l2_rho=2e-4)}


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_c1_sized_fast_100_steps(oracle_lib, precision):
    O = oracle_lib
    shape = (256, 256, 128)
    flags, rho, u = cases.block_case("urban", shape)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS["luw"]
    zones = dict(downstream_face=2, buffer_N=16, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=20, sponge_inv_tau=0.02)
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, 100, w, zones=zones)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, 100, w, arith=1, zones=zones, batched=True, expect_tiles=True)
    tol = TOL_C1_100[precision]
    e = H.errors(got, ref)
    H.report("c1_sized_fast_100_steps", precision=precision, steps=100, rel_l2_u=e[0], max_abs_u=e[1], rel_l2_rho=e[2], tol=tol)
    assert e[0] <= tol["rel_l2_u"] and e[1] <= tol["max_abs_u"] and e[2] <= tol["rel_l2_rho"], e


# ---------------------------------------------------------------------------------------------- relaxation zones: every downstream face, vertical nudging on / off
@pytest.mark.parametrize("tiled", [True, False], ids=["tile", "cell"])
@pytest.mark.parametrize("vertical", [0, 1], ids=["novert", "vert"])
@pytest.mark.parametrize("face", [0, 1, 2, 3, 4], ids=["none", "west", "east", "south", "north"])
def test_zone_variants_strict_equals_oracle(oracle_lib, monkeypatch, face, vertical, tiled):
    """FX/kernel.cpp:1523-1614 with every def_downstream_face and def_buffer_nudge_vertical (tests/test_oracle_vs_reference.py pins the oracle on the same grid)."""
    O = oracle_lib
    shape = (128, 20, 12)
    flags, rho, u = cases.urban(*shape, seed=9, edge=3, pitch=6)
    w = cases.relaxation_rate(1e-6)
    zones = dict(downstream_face=face, buffer_N=4, buffer_inv_tau=0.01, buffer_nudge_vertical=vertical, sponge_N=3, sponge_inv_tau=0.02)
    if not tiled:
        monkeypatch.setenv("LUW_NO_TILE", "1")
    for precision, arith in ((1, 0), (0, 0), (1, 1)):
        ref = H.run_cpu(O.Oracle(), O, shape, precision, H.FEATURE_SETS["luw"], flags, rho, u, 7, w, zones=zones)
        got = H.run_cuda(shape, precision, H.FEATURE_SETS["luw"], flags, rho, u, 7, w, arith=arith, zones=zones, expect_tiles=tiled)
        if arith == 0:
            assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision)), (precision, "DDFs differ")
            assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2]), (precision, "rho / u differ")
        else:
            e = H.errors(got, ref)
            assert e[0] <= 1e-3 and e[1] <= 2e-4, e


# ---------------------------------------------------------------------------------------------- decomposed runs (several domains on ONE GPU)
@pytest.mark.parametrize("D,arith", [((2, 2, 2), 0), ((1, 2, 2), 0), ((1, 2, 2), 1), ((1, 1, 4), 1), ((2, 2, 2), 1), ((2, 1, 1), 1)], ids=["2x2x2-strict", "1x2x2-strict", "1x2x2-fast", "1x1x4-fast", "2x2x2-fast", "2x1x1-fast"])
@pytest.mark.parametrize("precision", [0, 1], ids=["fp32", "fp16s"])
def test_decomposed_equals_single_domain(D, arith, precision):
    """D domains with halo exchange reproduce the single-domain run bit for bit (same kernels on both sides of the comparison)."""
    from latticeurbanwind_b200.lbm import LBM
    shape = (128, 24, 16)
    flags, rho, u = cases.urban(*shape, seed=21, edge=4, pitch=8)
    zones = dict(downstream_face=2, buffer_N=3, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=3, sponge_inv_tau=0.02)
    res = []
    for dd in ((1, 1, 1), D):
        lbm = LBM(shape, D=dd, nu=1e-6, precision=precision, features=H.FEATURE_SETS["luw"], arith=arith, f=H.FORCE, omega=H.OMEGA, **zones)
        lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
        lbm.run(7)
        lbm.read_from_device()
        res.append((lbm.rho.copy(), lbm.u.copy()))
        lbm.close()
    assert np.array_equal(res[0][0], res[1][0]), "rho differs between D=1 and the decomposed run"
    assert np.array_equal(res[0][1], res[1][1]), "u differs between D=1 and the decomposed run"


# ---------------------------------------------------------------------------------------------- dense host images <-> pitched device arrays
@pytest.mark.parametrize("Nx", [66, 64, 37], ids=["66-padded", "64-dense", "37-padded"])
def test_partial_uploads_and_downloads(Nx):
    """Memory<T>::enqueue_write_to_device / enqueue_read_from_device(offset, length) (FX/opencl.hpp:481-512) on element ranges that start and end
    inside rows and span components: the device rows are padded to multiples of 16 elements, host images are dense."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain
    Ny, Nz = 5, 4
    rng = np.random.default_rng(Nx)
    with Domain(Nx, Ny, Nz, precision=1, features=0, w=1.0, arith=0) as d:
        N = d.N
        full = rng.standard_normal(3 * N).astype(np.float32)
        d.u[:] = full
        d.write_to_device(A.FIELD_U)
        for off, cnt in [(0, 3 * N), (5, 7), (Nx - 3, 2 * Nx + 9), (N - 11, N + 30), (2 * N + Nx * 3, Nx * 4), (3 * N - 1, 1), (17, 0)]:
            d.u[:] = -1.0
            d.read_from_device(A.FIELD_U, off, cnt); d.finish_queue()
            assert np.array_equal(d.u[off:off + cnt], full[off:off + cnt]), (off, cnt)
            assert np.all(d.u[:off] == -1.0) and np.all(d.u[off + cnt:] == -1.0)
        patch = rng.standard_normal(3 * N).astype(np.float32)
        off, cnt = N - 2 * Nx - 5, 3 * Nx + 11  # crosses from ux into uy, ragged at both ends
        d.u[:] = patch
        d.write_to_device(A.FIELD_U, off, cnt)
        expect = full.copy(); expect[off:off + cnt] = patch[off:off + cnt]
        d.u[:] = 0.0
        d.read_from_device(A.FIELD_U); d.finish_queue()
        assert np.array_equal(d.u, expect)
        flags = rng.integers(0, 255, N).astype(np.uint8)
        d.flags[:] = flags
        d.write_to_device(A.FIELD_FLAGS)
        d.flags[:] = 0
        d.read_from_device(A.FIELD_FLAGS, 3, N - 7); d.finish_queue()
        assert np.array_equal(d.flags[3:N - 4], flags[3:N - 4])
        fi = rng.integers(0, 65535, 19 * N).astype(np.uint16)
        d.write_fi(fi)
        assert np.array_equal(d.read_fi(), fi)


# ---------------------------------------------------------------------------------------------- von Karman inlet (FX/kernel.cpp:2495-2571)
@pytest.mark.parametrize("arith", [0, 1], ids=["strict", "fast"])
@pytest.mark.parametrize("interp,t0,t1", [(0, 3.0, 4.0), (1, 3.0, 4.0), (1, 20000.0, 20001.0)], ids=["single", "interp", "interp-late"])
def test_vk_inlet_matches_oracle(oracle_lib, arith, interp, t0, t1):
    """u of the inlet cells = base + sigma * sum of modes. STRICT evaluates the reference's expression with CUDA's cosf (a few ulp from libm);
    FAST uses cos(a+b) = cos a cos b - sin a sin b with one range-reduced hardware sincos per mode (absolute error ~1e-6 per unit amplitude).
    Tolerance on u (lattice units, |u| ~ 0.1, sigma <= 0.004, 24 modes of amplitude ~1): 2e-7 STRICT, 1e-6 FAST; late in a run (phases of thousands of
    radians) the reference's own rounding of phase + phi to a float (<= 1.2e-4 rad per term) is what separates the two: 2e-5 FAST."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import Domain, VkInlet
    O = oracle_lib
    pc, pf, pd, md, M, V, N = H.vk_case()
    orc = O.Oracle().bind(O.make_params(*H.VK_SHAPE, O.FP16C, O.FEATURE_SETS["luw"]))
    ref = np.zeros(3 * N, np.float32)
    orc.vk_inlet_apply(interp, t0, t1, 0.25, pc, pf, pd, md, M, V, ref)
    with Domain(*H.VK_SHAPE, precision=2, features=H.FEATURE_SETS["luw"], w=1.0, arith=arith, **H.ZONES) as d:
        d.u[:] = 0.0
        d.write_to_device(A.FIELD_U)
        vk = VkInlet(d, pc, pf, pd, md, M, V)
        vk.apply(interp, t0, t1, 0.25)
        d.read_from_device(A.FIELD_U); d.finish_queue()
        vk.close()
        err = float(np.abs(d.u - ref).max())
        assert err <= (2e-7 if arith == 0 else 1e-6 if t0 < 1000.0 else 2e-5), err
        untouched = np.ones(3 * N, bool)
        for c in range(3):
            untouched[c * N + pc.astype(np.int64)] = False
        assert np.all(d.u[untouched] == 0.0)


# ---------------------------------------------------------------------------------------------- full-size properties (no oracle at these sizes)
def test_full_size_decomposition_identity_and_fixed_point():
    """At a bench-sized block (33.5 M cells, the urban case of BASELINE configs[2] at a quarter of its footprint) the oracle takes minutes, so parity is carried by
    size-independent properties: (1) the 1x2x2 decomposition (four domains sharing the GPU, halo exchange in the library) reproduces the single-domain
    FAST FP16S run bit for bit; (2) cells the step must not touch (TYPE_S buildings and ground) keep rho / u / flags; (3) u stays inside the clamp +-c."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.lbm import LBM
    shape = (512, 512, 128)
    flags, rho, u = cases.block_case("urban", shape)
    zones = dict(downstream_face=2, buffer_N=16, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=20, sponge_inv_tau=0.02)
    res = []
    for D in ((1, 1, 1), (1, 2, 2)):
        lbm = LBM(shape, D=D, nu=1e-6, precision=A.FP16S, features=H.FEATURE_SETS["luw"], arith=A.ARITH_FAST, omega=H.OMEGA, **zones)
        lbm.flags[:], lbm.rho[:], lbm.u[:] = flags, rho, u
        lbm.run(12)
        lbm.read_from_device()
        res.append((lbm.rho.copy(), lbm.u.copy(), lbm.flags.copy()))
        lbm.close()
    assert np.array_equal(res[0][0], res[1][0]), "rho differs between D=1 and 1x2x2"
    assert np.array_equal(res[0][1], res[1][1]), "u differs between D=1 and 1x2x2"
    r1, u1, f1 = res[0]
    assert np.array_equal(f1, flags)
    solid = (flags & 3) == 1
    assert solid.sum() > 100000
    N = flags.size
    assert np.array_equal(r1[solid], rho[solid])
    for c in range(3):
        assert np.all(u1[c * N:(c + 1) * N][solid] == 0.0)  # initialize zeroes u in solids (FX/kernel.cpp:1379), the step never writes them
    assert float(np.abs(u1).max()) <= 0.57735027 + 1e-7 and np.isfinite(r1).all()
    fluid = ~solid & ((flags & 3) != 2)
    lo, hi = float(r1[fluid].min()), float(r1[fluid].max())  # impulsive start against the cubes: a pressure wave of order rho*u/c_s = 0.17
    assert 0.6 < lo and hi < 1.5, (lo, hi)


def test_cell_sets_move_boundary_data_without_whole_fields():
    """luw_cellset_upload / _download (boundary-field upload and probe read-back, SURVEY.md 8-a18): several uploads and read-backs in flight on the copy
    stream, staging slots reused, results equal to plain whole-field transfers."""
    from latticeurbanwind_b200 import _cabi as A
    from latticeurbanwind_b200.domain import CellSet, Domain, pinned_empty
    Nx, Ny, Nz = 66, 9, 7
    rng = np.random.default_rng(11)
    with Domain(Nx, Ny, Nz, precision=1, features=0, w=1.0, arith=0) as d:
        N = d.N
        base = rng.standard_normal(3 * N).astype(np.float32)
        d.u[:] = base
        d.rho[:] = rng.standard_normal(N).astype(np.float32)
        rho0 = d.rho.copy()
        d.upload_all()
        cells = rng.choice(N, 500, replace=False).astype(np.uint64)
        cs = CellSet(d, cells)
        want = base.copy()
        bufs = []
        for k in range(5):  # five uploads back to back: the last one wins, none may be torn
            b = pinned_empty(3 * cs.count, np.float32)
            b[:] = rng.standard_normal(3 * cs.count).astype(np.float32)
            bufs.append(b)
            cs.upload(A.FIELD_U, b)
        for c in range(3):
            want[c * N + cells.astype(np.int64)] = bufs[-1][c * cs.count:(c + 1) * cs.count]
        outs = [(pinned_empty(3 * cs.count, np.float32), pinned_empty(cs.count, np.float32)) for _ in range(3)]
        for ou, orr in outs:  # three read-back pairs in flight
            cs.download(A.FIELD_U, ou); cs.download(A.FIELD_RHO, orr)
        d.finish_queue()
        for ou, orr in outs:
            assert np.array_equal(ou, bufs[-1]) and np.array_equal(orr, rho0[cells.astype(np.int64)])
        d.read_from_device(A.FIELD_U); d.finish_queue()
        assert np.array_equal(d.u, want)
        cs.close()


@pytest.mark.parametrize("precision,arith", [(2, 0), (2, 1), (1, 1)], ids=["fp16c-strict", "fp16c-fast", "fp16s-fast"])
def test_reference_example_lattice_runs_the_tile_kernel(oracle_lib, precision, arith):
    """253 x 250 x 59 is the lattice of the reference's own example deck (examples/example_ProfileResearch_noDEM at its default cell size): odd Nx, partial tiles
    in x, y and z. It must reach the TMA tile kernel (luw_domain_step_kernel == 1) and equal the oracle."""
    O = oracle_lib
    shape = (253, 250, 59)
    flags, rho, u = cases.block_case("urban", shape)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS["luw"]
    zones = dict(downstream_face=2, buffer_N=16, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=20, sponge_inv_tau=0.02)
    ref = H.run_cpu(O.Oracle(), O, shape, precision, feat, flags, rho, u, 6, w, zones=zones)
    got = H.run_cuda(shape, precision, feat, flags, rho, u, 6, w, arith=arith, zones=zones, batched=True, expect_tiles=True)
    if arith == 0:
        assert np.array_equal(H.decode(O, None, got[0], precision), H.decode(O, None, ref[0], precision)), "DDFs differ"
        assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2]), "rho / u differ"
    else:
        e = H.errors(got, ref)
        assert e[0] <= 1e-3 and e[1] <= 2e-4, e


def test_c1_sized_case_equals_oracle(oracle_lib):
    """BASELINE configs[0] scale (256 x 256 x 128 = 8.4 M cells, FP32, SRT + Smagorinsky, equilibrium inflow on five faces, bounce-back cubes, Coriolis,
    nudging, sponge -- the profile case's physics on the synthetic block array): 10 steps, STRICT arithmetic, every rho / u value equal to the oracle's."""
    O = oracle_lib
    shape = (256, 256, 128)
    flags, rho, u = cases.block_case("urban", shape)
    w = cases.relaxation_rate(1e-6)
    feat = H.FEATURE_SETS["luw"]
    zones = dict(downstream_face=2, buffer_N=16, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=20, sponge_inv_tau=0.02)
    ref = H.run_cpu(O.Oracle(), O, shape, 0, feat, flags, rho, u, 10, w, zones=zones)
    got = H.run_cuda(shape, 0, feat, flags, rho, u, 10, w, arith=0, zones=zones, batched=True, expect_tiles=True)
    assert np.array_equal(got[1], ref[1]), "rho differs"
    assert np.array_equal(got[2], ref[2]), "u differs"
    fast = H.run_cuda(shape, 0, feat, flags, rho, u, 10, w, arith=1, zones=zones, batched=True, expect_tiles=True)
    assert H.rel_l2(fast[2], ref[2]) <= 1e-5 and float(np.abs(fast[2] - ref[2]).max()) <= 2e-6  # SURVEY 8c: FP32 rel-L2(u) <= 1e-5, max-abs(u) <= 2e-6
