"""One stream_collide step, element by element, against the float64 reference (oracle/step_f64.py).

The FAST kernels (the lean loop V5 / V6, the two-pass and single-pass tile kernels, the per-cell kernel) regroup the collision and use approximate reciprocals
and square roots, so they cannot equal the oracle bit for bit; the multi-step parity tests hold them to rho / u bars set by many steps of flow. Here one step
from a hand-built state is compared per DDF with a float64 restatement, at bars tied to float rounding:
  * image elements the step does not store: bit-identical to the input;
  * stored elements, FP32: |dev - ref| <= K * 2^-24 * s_e, s_e = |f_in| + |f_eq| + w_i of the element;
  * stored elements, FP16S / FP16C: the correctly rounded code of the float64 value, except where that value lies within eps = K * 2^-24 * s_e of a rounding
    midpoint, where either neighbour is accepted (the exempted fraction is reported and bounded);
  * rho / u written by the step (UPDATE_FIELDS) and by update_fields: within K_RU * 2^-24 of the float64 value, relative to the magnitudes summed into them.
    These never pass through the 16-bit codecs, so the bar is the same for every storage format.
STRICT arithmetic meets the same bars; its bit-exactness against the oracle is tested elsewhere.

The CPU tests pin the reference against the C oracle (float32 STRICT) and show that the bars separate known defects by a wide margin.
"""
import functools

import numpy as np
import pytest

from latticeurbanwind_b200 import cases
from oracle import step_f64 as S
from tests import helpers as H

ULP = 2.0 ** -24
# FEAT (the template bits of the step kernels) -> the feature set a test runs; 14 / 15 carry the relaxation zones (run-time branches of the same instantiations)
FEATURES = {0: 0, 4: 4, 5: 5, 14: 62, 15: 63}
W_LES = float(cases.relaxation_rate(1e-6))
FORCE = (2e-4, -1e-4, 3e-4)  # larger than a deck's, so that the Guo term and the Coriolis force stand well above float rounding
OMEGA = (1e-3, 2e-3, 3e-3)
ZONES = dict(downstream_face=2, buffer_N=3, buffer_inv_tau=0.01, buffer_nudge_vertical=1, sponge_N=2, sponge_inv_tau=0.02)
# Bars, in units of 2^-24 of the element's scale, at about twice the largest error measured on a B200 over every case below (DESIGN.md section 4,
# profiles/step_f64_parity_measured.jsonl): FP32 DDFs 11.4, FP16S / FP16C the eps the device's codes need 3.9 / 5.4, rho / u 2.9. The C oracle's float32 STRICT
# step (the CPU tests) measures 8.4 / 4.1 / 2.9 and 2.1: the floor of float rounding, which every kernel has to meet as well.
K_DDF = {0: 24.0, 1: 8.0, 2: 12.0}
K_RU = 6.0
MAX_EXEMPT = {0: 0.0, 1: 0.06, 2: 0.15}  # fraction of stored FP16 elements within eps of a rounding midpoint
SEPARATION = 30.0


# ---------------------------------------------------------------------------------------------- storage formats
def encode(v, precision):
    """float64 -> DDF storage through float32, as the C oracle stores: FP32 as is, FP16S = half(32768 f) round-to-nearest-even, FP16C = luwo_float_to_fp16c."""
    x = np.asarray(v, np.float64).astype(np.float32)
    if precision == 0:
        return x
    if precision == 1:
        return (x * np.float32(32768.0)).astype(np.float16).view(np.uint16)
    b = (x.view(np.uint32).astype(np.int64) + 0x800) & 0xFFFFFFFF
    e, m = (b & 0x7F800000) >> 23, b & 0x007FFFFF
    r = (b & 0x80000000) >> 16
    r |= np.where(e > 112, (((e - 112) << 11) & 0x7800) | (m >> 12), 0)
    r |= np.where((e < 113) & (e > 100), (((0x007FF800 + m) >> np.clip(124 - e, 0, 31)) + 1) >> 1, 0)
    return r.astype(np.uint16)


@functools.lru_cache(maxsize=None)
def _table(precision):
    from oracle import wall_loads_oracle as WL
    return WL.decode(np.arange(65536, dtype=np.uint16), precision).astype(np.float64)


def decode(img, precision):
    return np.asarray(img, np.float64) if precision == 0 else _table(precision)[np.asarray(img, np.uint16)]


@functools.lru_cache(maxsize=None)
def _grid(precision):
    """(the format's finite values ascending, the midpoints between neighbours)."""
    t = _table(precision)
    V = np.unique(t[np.isfinite(t)])
    return V, 0.5 * (V[:-1] + V[1:])


def code_check(got, ref, eps, precision):
    """FP16: (ok, exempt, k_needed) per element. ok: the decoded device value is a code that some x in [ref - eps, ref + eps] rounds to; exempt: that interval
    holds a midpoint; k_needed: the eps (in units of the caller's scale) the element needs, 0 where it holds the correctly rounded code."""
    V, mids = _grid(precision)
    d = np.searchsorted(V, got)
    assert np.array_equal(V[np.minimum(d, V.size - 1)], got), "device value is not a code of the format"
    r = np.searchsorted(mids, ref)
    lo, hi = np.searchsorted(mids, ref - eps), np.searchsorted(mids, ref + eps)
    top = mids.size - 1
    need = np.where(d == r, 0.0, np.where(d > r, mids[np.clip(d - 1, 0, top)] - ref, ref - mids[np.clip(d, 0, top)]))
    return (lo <= d) & (d <= hi), lo != hi, need


def ddf_errors(got_img, in_img, ref, precision, k):
    """Compares a post-step image with the reference. Returns a dict of measured values and the list of failing elements (flat index, measured k)."""
    unwritten = ~ref.written
    stale_ok = np.array_equal(got_img[unwritten].view(np.uint32 if precision == 0 else np.uint16), in_img[unwritten].view(np.uint32 if precision == 0 else np.uint16))
    idx = np.flatnonzero(ref.written)
    got = decode(got_img[idx], precision)
    want, s = ref.fi[idx], ref.scale[idx]
    if precision == 0:
        kk = np.abs(got - want) / (ULP * s)
        ok, exempt = kk <= k, np.zeros(idx.size, bool)
    else:
        ok, exempt, need = code_check(got, want, k * ULP * s, precision)
        kk = need / (ULP * s)
    bad = idx[~ok]
    return dict(unwritten_identical=bool(stale_ok), k_max=float(kk.max()) if kk.size else 0.0, exempt=float(exempt.mean()) if exempt.size else 0.0,
                stored=int(idx.size)), [(int(i), float(v)) for i, v in zip(bad[:8], kk[~ok][:8])]


def field_scales(p, fi64, flags, t, u_ref):
    """Per-cell magnitudes summed into rho and u: s_rho = 1 + sum |f_i|, s_u_a = sum |c_ia f_i| / rho + |u_a| (dense, zero where the step does not run)."""
    N = flags.size
    cells = S.executes(p, flags)
    fin = fi64[S.ddf_locations(p, cells, t)]
    a = np.abs(fin)
    s_rho = np.zeros(N)
    s_rho[cells] = 1.0 + a.sum(0)
    rho = np.abs(fin.sum(0) + 1.0)
    s_u = np.zeros(3 * N)
    for c, cc in enumerate((S.CX, S.CY, S.CZ)):
        s_u[c * N + cells] = (np.abs(cc)[:, None] * a).sum(0) / rho + np.abs(u_ref[c * N + cells])
    return s_rho, s_u


def field_errors(got_rho, got_u, in_rho, in_u, ref_rho, ref_u, s_rho, s_u):
    """(k_max over the values the reference changes, whether the others keep their bits, worst value)."""
    out = []
    same = True
    worst = None
    for got, inp, ref, s in ((got_rho, in_rho, ref_rho, s_rho), (got_u, in_u, ref_u, s_u)):
        keep = ref == inp.astype(np.float64)  # not written: must keep its bits
        same &= bool(np.array_equal(got[keep].view(np.uint32), inp[keep].view(np.uint32)))
        live = ~keep
        k = np.zeros(got.size)
        k[live] = np.abs(got[live] - ref[live]) / (ULP * s[live])
        out.append(float(k.max()) if k.size else 0.0)
        i = int(np.argmax(k))
        if worst is None or k[i] > worst[1]:
            worst = (("rho" if got is got_rho else "u"), int(i), float(k[i]))
    return max(out), same, worst


# ---------------------------------------------------------------------------------------------- the hand-built state
def _fields(shape, layout, rng):
    """flags, rho, u: 'walled' = ground TYPE_S, TYPE_E on x = 0 / Nx-1, y = 0 / Ny-1 and the top (the faces the relaxation zones read), 'box' = periodic; both
    with scattered TYPE_S and TYPE_G cells inside. rho / u are boundary values (TYPE_E) or stale fields, independent of what the cells stream in."""
    Nx, Ny, Nz = shape
    N = Nx * Ny * Nz
    n = np.arange(N)
    x, y, z = n % Nx, (n // Nx) % Ny, n // (Nx * Ny)
    flags = np.zeros(N, np.uint8)
    if layout == "walled":
        flags[(x == 0) | (x == Nx - 1) | (y == 0) | (y == Ny - 1) | (z == Nz - 1)] = S.TYPE_E
        flags[z == 0] = S.TYPE_S
    pick = rng.random(N)
    inner = flags == 0
    flags[inner & (pick < 0.05)] = S.TYPE_S
    flags[inner & (pick >= 0.05) & (pick < 0.08)] = S.TYPE_G
    rho = (1.0 + 0.05 * (2.0 * rng.random(N) - 1.0)).astype(np.float32)
    u = (0.1 * (2.0 * rng.random(3 * N) - 1.0)).astype(np.float32)
    return flags, rho, u


def _populations(N, rng):
    """float64 [19, N]: what each cell streams in -- the equilibrium of rho in 1 +- 0.05, |u_a| <= 0.2, plus a non-equilibrium part of 3 % of w_i; special
    cells: exact equilibrium (5 %), |u_x| = 0.75 > c (3 %), rho = 0.7 and rho = 1.4 (2 % each)."""
    rho = 1.0 + 0.05 * (2.0 * rng.random(N) - 1.0)
    u = 0.2 * (2.0 * rng.random((3, N)) - 1.0)
    kind = rng.random(N)
    u[0] = np.where((kind >= 0.05) & (kind < 0.08), np.sign(u[0]) * 0.75, u[0])
    rho = np.where((kind >= 0.08) & (kind < 0.10), 0.7, np.where((kind >= 0.10) & (kind < 0.12), 1.4, rho))
    neq = 0.03 * S.W[:, None] * (2.0 * rng.random((19, N)) - 1.0)
    neq[:, kind < 0.05] = 0.0
    return S.f_eq(rho, u[0], u[1], u[2]) + neq


@functools.lru_cache(maxsize=None)
def make_case(shape, layout, precision, feat, t, D=(1, 1, 1), block=(0, 0, 0), zones=tuple(sorted(ZONES.items())), seed=0):
    """(params, flags, rho, u, image, reference Step). `shape`: the lattice, or for D != (1,1,1) the global lattice of which block `block` is taken."""
    from oracle import oracle as O
    rng = np.random.default_rng([seed, *shape, precision, feat, t, *block])
    if D == (1, 1, 1):
        Ov = (0, 0, 0)
        flags, rho, u = _fields(shape, layout, rng)
        local = shape
    else:
        flags, rho, u = _fields(shape, layout, rng)
        local, Ov, flags, rho, u = H.cut_block(shape, D, block, flags, rho, u)
    p = O.make_params(*local, precision, FEATURES[feat], w=W_LES, D=D, O=Ov, **dict(zones))
    N = int(np.prod(local))
    img = np.zeros(19 * N, np.float32 if precision == 0 else np.uint16)
    img[S.ddf_locations(p, np.arange(N), t)] = encode(_populations(N, rng), precision)
    ref = S.stream_collide(decode(img, precision), flags, rho, u, p, t, FORCE, OMEGA)
    return p, flags, rho, u, img, ref


# ---------------------------------------------------------------------------------------------- CPU: the reference against the C oracle, and the bars' reach
def test_encode_matches_the_c_codecs(oracle_lib):
    O = oracle_lib
    orc = O.Oracle()
    x = H.codec_sweep()
    x = x[np.abs(x) < 60000.0 / 32768.0]
    assert np.array_equal(encode(x, 1), np.array([orc.float_to_half(np.float32(v) * np.float32(32768.0)) for v in x], np.uint16))
    assert np.array_equal(encode(x, 2), np.array([orc.float_to_fp16c(v) for v in x], np.uint16))


def _oracle_step(O, p, flags, rho, u, img, t):
    fi, r, uu = img.copy(), rho.copy(), u.copy()
    O.Oracle().bind(p).stream_collide(fi, r, uu, flags, t, FORCE, OMEGA)
    return fi, r, uu


CPU_CASES = {"box": ((16, 10, 8), "box", (1, 1, 1), (0, 0, 0)), "urban-oddNx": ((25, 12, 9), "walled", (1, 1, 1), (0, 0, 0)),
             "cut2x2x2": ((28, 20, 14), "walled", (2, 2, 2), (1, 0, 1))}


@pytest.mark.parametrize("t", [0, 1], ids=["even", "odd"])
@pytest.mark.parametrize("feat", [0, 4, 5, 14, 15], ids=lambda f: f"FEAT{f}")
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("where", list(CPU_CASES))
def test_f64_step_matches_the_c_oracle(oracle_lib, where, precision, feat, t):
    """The C oracle (float32, pinned to the reference's kernel text) against the float64 restatement: elements the reference does not store are untouched,
    stored ones and rho / u agree within float32 rounding (the STRICT floor, recorded)."""
    if where == "box" and feat != 0:
        pytest.skip("a periodic box has no faces for the boundary cells and relaxation zones")
    shape, layout, D, block = CPU_CASES[where]
    p, flags, rho, u, img, ref = make_case(shape, layout, precision, feat, t, D, block)
    fi, r, uu = _oracle_step(oracle_lib, p, flags, rho, u, img, t)
    m, bad = ddf_errors(fi, img, ref, precision, K_DDF[precision])
    s_rho, s_u = field_scales(p, decode(img, precision), flags, t, ref.u)
    k_ru, same, worst = field_errors(r, uu, rho, u, ref.rho, ref.u, s_rho, s_u)
    H.report("step_f64_strict_floor", where=where, precision=precision, feat=feat, t=t, k_ru=k_ru, **m)
    assert m["unwritten_identical"], "the oracle changed an element the reference does not store"
    assert not bad and m["exempt"] <= MAX_EXEMPT[precision], (m, bad)
    assert same and k_ru <= K_RU, (k_ru, worst)


@pytest.mark.parametrize("vertical", [0, 1], ids=["novert", "vert"])
@pytest.mark.parametrize("face", [0, 1, 2, 3, 4], ids=["none", "west", "east", "south", "north"])
def test_f64_zones_match_the_c_oracle(oracle_lib, face, vertical):
    """Buffer nudging at every downstream face, vertical nudging on and off, with the top sponge: FP32, FEAT 15."""
    zones = dict(ZONES, downstream_face=face, buffer_nudge_vertical=vertical, buffer_N=4, sponge_N=3)
    p, flags, rho, u, img, ref = make_case((25, 14, 11), "walled", 0, 15, face % 2, zones=tuple(sorted(zones.items())))
    fi, r, uu = _oracle_step(oracle_lib, p, flags, rho, u, img, face % 2)
    m, bad = ddf_errors(fi, img, ref, 0, K_DDF[0])
    s_rho, s_u = field_scales(p, decode(img, 0), flags, face % 2, ref.u)
    k_ru, same, worst = field_errors(r, uu, rho, u, ref.rho, ref.u, s_rho, s_u)
    assert m["unwritten_identical"] and not bad and same and k_ru <= K_RU, (m, bad, k_ru, worst)


def test_f64_update_fields_matches_the_c_oracle(oracle_lib):
    O = oracle_lib
    for precision in (0, 1, 2):
        for feat in (4, 15):
            p, flags, rho, u, img, ref = make_case((25, 12, 9), "walled", precision, feat, 1)
            r, uu = rho.copy(), u.copy()
            O.Oracle().bind(p).update_fields(img, r, uu, flags, 1, FORCE, OMEGA)
            rr, ur = S.update_fields(decode(img, precision), flags, rho, u, p, 1, FORCE, OMEGA)
            s_rho, s_u = field_scales(p, decode(img, precision), flags, 1, ur)
            k_ru, same, worst = field_errors(r, uu, rho, u, rr, ur, s_rho, s_u)
            assert same and k_ru <= K_RU, (precision, feat, k_ru, worst)


DEFECTS = ["stale_slot", "swapped_parity", "no_smagorinsky", "no_forcing", "partner_rhom1"]


@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("defect", DEFECTS)
def test_bars_separate_known_defects(oracle_lib, defect, precision):
    """Each defect moves at least one stored element by >= SEPARATION times the FAST bar (for a stale slot: in every direction), and the 16-bit code check flags it."""
    t = 1
    p, flags, rho, u, img, ref = make_case((25, 12, 9), "walled", precision, 15, t)
    fi64 = decode(img, precision)
    if defect == "stale_slot":
        bad = fi64.copy()
        idx = np.flatnonzero(ref.written)
        slot = idx // flags.size
        k = np.abs(fi64[idx] - ref.fi[idx]) / (K_DDF[precision] * ULP * ref.scale[idx])
        bad_ratio = min(float(k[slot == i].max()) for i in range(19))
    else:
        if defect == "swapped_parity":
            bad = S.stream_collide(fi64, flags, rho, u, p, t ^ 1, FORCE, OMEGA).fi
        elif defect == "no_smagorinsky":
            q = oracle_lib.make_params(p.Nx, p.Ny, p.Nz, precision, FEATURES[15] & ~S.SUBGRID, w=W_LES, **ZONES)
            bad = S.stream_collide(fi64, flags, rho, u, q, t, FORCE, OMEGA).fi
        else:
            bad = S.stream_collide(fi64, flags, rho, u, p, t, FORCE, OMEGA, defect=defect).fi
        idx = np.flatnonzero(ref.written)
        bad_ratio = float((np.abs(bad[idx] - ref.fi[idx]) / (K_DDF[precision] * ULP * ref.scale[idx])).max())
    flagged = None
    if precision > 0:
        idx = np.flatnonzero(ref.written)
        ok, _, _ = code_check(decode(encode(bad[idx], precision), precision), ref.fi[idx], K_DDF[precision] * ULP * ref.scale[idx], precision)
        flagged = int((~ok).sum())
    H.report("step_f64_bar_separation", defect=defect, precision=precision, ratio=bad_ratio, fp16_flagged=flagged)
    assert bad_ratio >= SEPARATION, bad_ratio
    assert flagged is None or flagged > 0


# ---------------------------------------------------------------------------------------------- GPU: every step kernel against the reference
def run_device(case, precision, feat, t, arith, monkeypatch, variant=None, no_tile=False, expect_tiles=True):
    from latticeurbanwind_b200.domain import Domain
    p, flags, rho, u, img, ref = case
    if variant is None:
        monkeypatch.delenv("LUW_TILE_VARIANT", raising=False)
    else:
        monkeypatch.setenv("LUW_TILE_VARIANT", str(variant))
    if no_tile:
        monkeypatch.setenv("LUW_NO_TILE", "1")
    else:
        monkeypatch.delenv("LUW_NO_TILE", raising=False)
    zones = dict(downstream_face=p.downstream_face, buffer_N=p.buffer_N, buffer_inv_tau=p.buffer_inv_tau, buffer_nudge_vertical=p.buffer_nudge_vertical,
                 sponge_N=p.sponge_N, sponge_inv_tau=p.sponge_inv_tau)
    with Domain(int(p.Nx), int(p.Ny), int(p.Nz), D=(p.Dx, p.Dy, p.Dz), O=(p.Ox, p.Oy, p.Oz), precision=precision, features=FEATURES[feat], w=W_LES,
                arith=arith, **zones) as d:
        assert d.uses_tiles() == expect_tiles, "unexpected stream_collide implementation"
        d.rho[:], d.u[:], d.flags[:] = rho, u, flags
        d.upload_all()
        d.write_fi(img)
        d.f, d.omega = FORCE, OMEGA
        d.t = t
        d.enqueue_stream_collide()
        fi = d.read_fi()
        d.download_all()
        r1, u1 = d.rho.copy(), d.u.copy()
        d.t = t + 1
        d.enqueue_update_fields()
        d.download_all()
        return fi, r1, u1, d.rho.copy(), d.u.copy()


def check_device(name, case, precision, feat, t, got, **tags):
    p, flags, rho, u, img, ref = case
    fi, r1, u1, r2, u2 = got
    m, bad = ddf_errors(fi, img, ref, precision, K_DDF[precision])
    s_rho, s_u = field_scales(p, decode(img, precision), flags, t, ref.u)
    k_sc, same_sc, worst_sc = field_errors(r1, u1, rho, u, ref.rho, ref.u, s_rho, s_u)
    # update_fields on the device's own post-step image: isolates that kernel's moments from the step's rounding
    rr, ur = S.update_fields(decode(fi, precision), flags, r1, u1, p, t + 1, FORCE, OMEGA)
    s_rho2, s_u2 = field_scales(p, decode(fi, precision), flags, t + 1, ur)
    k_uf, same_uf, worst_uf = field_errors(r2, u2, r1, u1, rr, ur, s_rho2, s_u2)
    H.report(name, precision=precision, feat=feat, t=t, k_ru_step=k_sc, k_ru_update=k_uf, **m, **tags)
    N = flags.size
    where = [dict(slot=i // N, cell=i % N, xyz=(i % N % int(p.Nx), i % N // int(p.Nx) % int(p.Ny), i % N // (int(p.Nx) * int(p.Ny))),
                  flag=int(flags[i % N]), k=k) for i, k in bad]
    assert m["unwritten_identical"], "an element the step must not store was changed"
    assert not where, f"stored DDFs off the float64 reference (first {len(where)}): {where}"
    assert m["exempt"] <= MAX_EXEMPT[precision], m
    assert same_sc and k_sc <= K_RU, ("rho / u after stream_collide", k_sc, worst_sc)
    assert same_uf and k_uf <= K_RU, ("rho / u after update_fields", k_uf, worst_uf)


VARIANT_SHAPE = (259, 9, 6)  # odd Nx wider than every tile (FP32 V3 is 256 wide), padded row pitch, partial tiles in x, y and z
TILED_SHAPES = [(64, 8, 4), (128, 20, 12), (80, 10, 7), (192, 9, 5), (768, 6, 4), (66, 10, 6), (130, 7, 5), (202, 6, 4), (65, 8, 4), (129, 7, 5), (253, 10, 7), (385, 5, 3)]


def _layout(feat):
    return "box" if feat == 0 else "walled"


@pytest.mark.gpu
@pytest.mark.parametrize("t", [0, 1], ids=["even", "odd"])
@pytest.mark.parametrize("variant", [None, 0, 1, 2, 3, 4, 5, 6, 7], ids=lambda v: "default" if v is None else f"V{v}")
@pytest.mark.parametrize("feat", [0, 4, 5, 14, 15], ids=lambda f: f"FEAT{f}")
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_fast_step_every_variant(monkeypatch, precision, feat, variant, t):
    case = make_case(VARIANT_SHAPE, _layout(feat), precision, feat, t)
    got = run_device(case, precision, feat, t, 1, monkeypatch, variant=variant)
    check_device("step_f64_fast_variant", case, precision, feat, t, got, variant=-1 if variant is None else variant)


@pytest.mark.gpu
@pytest.mark.parametrize("t", [0, 1], ids=["even", "odd"])
@pytest.mark.parametrize("feat", [4, 15], ids=lambda f: f"FEAT{f}")
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("shape", TILED_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_fast_step_tiled_shapes(monkeypatch, shape, precision, feat, t):
    case = make_case(shape, _layout(feat), precision, feat, t)
    got = run_device(case, precision, feat, t, 1, monkeypatch)
    check_device("step_f64_fast_shape", case, precision, feat, t, got, shape="x".join(map(str, shape)))


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [1, 0], ids=["fast", "strict"])
@pytest.mark.parametrize("t", [0, 1], ids=["even", "odd"])
@pytest.mark.parametrize("feat", [0, 4, 5, 14, 15], ids=lambda f: f"FEAT{f}")
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
@pytest.mark.parametrize("kernel", ["narrow", "no-tile"])
def test_step_per_cell_kernel(monkeypatch, kernel, precision, feat, t, arith):
    """k_stream_collide: a lattice narrower than the 64-wide tiles, and LUW_NO_TILE=1 on a tileable one."""
    shape = (37, 9, 6) if kernel == "narrow" else (129, 7, 5)
    case = make_case(shape, _layout(feat), precision, feat, t)
    got = run_device(case, precision, feat, t, arith, monkeypatch, no_tile=kernel == "no-tile", expect_tiles=False)
    check_device("step_f64_per_cell", case, precision, feat, t, got, kernel=kernel, arith=arith)


@pytest.mark.gpu
@pytest.mark.parametrize("t", [0, 1], ids=["even", "odd"])
@pytest.mark.parametrize("feat", [0, 4, 5, 14, 15], ids=lambda f: f"FEAT{f}")
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_strict_step_meets_the_same_bars(monkeypatch, precision, feat, t):
    case = make_case(VARIANT_SHAPE, _layout(feat), precision, feat, t)
    got = run_device(case, precision, feat, t, 0, monkeypatch)
    check_device("step_f64_strict", case, precision, feat, t, got)


@pytest.mark.gpu
@pytest.mark.parametrize("arith", [1, 0], ids=["fast", "strict"])
@pytest.mark.parametrize("t", [0, 1], ids=["even", "odd"])
@pytest.mark.parametrize("feat", [0, 4, 5, 14, 15], ids=lambda f: f"FEAT{f}")
@pytest.mark.parametrize("precision", [0, 1, 2], ids=["fp32", "fp16s", "fp16c"])
def test_step_decomposed_block(monkeypatch, precision, feat, t, arith):
    """Block (1, 0, 1) of a 2x2x2 cut, 128 cells wide with its halo columns: halo cells do not run, their elements that owned cells do not store survive."""
    case = make_case((252, 12, 10), "walled", precision, feat, t, D=(2, 2, 2), block=(1, 0, 1))
    assert (int(case[0].Nx), int(case[0].Ny), int(case[0].Nz)) == (128, 8, 7)
    got = run_device(case, precision, feat, t, arith, monkeypatch)
    check_device("step_f64_decomposed", case, precision, feat, t, got, arith=arith)
