"""TEST INFRASTRUCTURE: one stream_collide step (and update_fields) of oracle/luw_oracle.c (stream_collide_impl / update_fields_impl, FX/kernel.cpp:1475-1780,
1938-2028) restated in numpy float64, vectorised over cells. Only tests/ may import this; the product path never does.

It is the high-precision reference the FAST kernels are held against element by element: the same formulas, with the float32 constants and parameters the
device receives (weights, def_c, 1/3, the Smagorinsky constant, w, inv_tau values, force, omega) promoted to double, and every operation in double --
including the sin^2 ramps of the relaxation zones, which the device reads from host-built float tables. What remains between this reference and a kernel is
the kernel's own float rounding.

  ddf_locations   [19, K] flat indices i*N + n of the image elements cell n loads (and stores back) at parity t&1: Esoteric-Pull (FX/kernel.cpp:1338-1351)
  executes        cells the step runs: not a halo cell of a decomposed block, not TYPE_S, not TYPE_G
  f_eq            the shifted D3Q19 equilibrium (the DDFs are stored as f - w_i)
  stream_collide  -> Step(fi, rho, u, written, scale): the post-step image in float64, rho / u after the UPDATE_FIELDS writes, the mask of image elements
                  an executing cell stores, and each stored element's scale |f_in| + |f_eq| + w_i (what its rounding error is measured against)
  update_fields   -> (rho, u) as the update_fields kernel leaves them

Inputs: the DDF image decoded to float64 (fi[i*N + n], dense host layout n = x + (y + z*Ny)*Nx), flags, rho, u (u = [ux | uy | uz]) and an oracle.Params.
The relaxation zones read u of the face / top-row cells from the input fields, which is what a kernel reads when those cells do not write u in the same
step (TYPE_E or TYPE_S faces, as every LUW deck and test case has them).
"""
from collections import namedtuple

import numpy as np

F32, F64 = np.float32, np.float64
UPDATE_FIELDS, VOLUME_FORCE, EQUILIBRIUM_BOUNDARIES, SUBGRID, BUFFER_NUDGING, TOP_SPONGE = 1, 2, 4, 8, 16, 32
TYPE_S, TYPE_E, TYPE_BO, TYPE_G, TYPE_SU = 0x01, 0x02, 0x03, 0x20, 0x38
# c_i in the DDF order of the kernels (lbm_common.cuh neighbors(): j[i] = n + c_i)
CX = np.array([0, 1, -1, 0, 0, 0, 0, 1, -1, 1, -1, 0, 0, 1, -1, 1, -1, 0, 0])
CY = np.array([0, 0, 0, 1, -1, 0, 0, 1, -1, 0, 0, 1, -1, -1, 1, 0, 0, 1, -1])
CZ = np.array([0, 0, 0, 0, 0, 1, -1, 0, 0, 1, -1, 1, -1, 0, 0, -1, 1, -1, 1])
# the float32 constants of the kernels (FX/lbm.cpp:662, 672-674; FX/kernel.cpp:1103-1113, 1735), promoted
W = np.array([F32(1.0) / F32(3.0)] + [F32(1.0) / F32(18.0)] * 6 + [F32(1.0) / F32(36.0)] * 12, F64)
LAT_C = F64(F32(0.57735027))
THIRD = F64(F32(0.33333334))
SMAG = F64(F32(0.76421222))
HALF_PI = F64(F32(1.5707963267948966))

Step = namedtuple("Step", "fi rho u written scale")


def _coords(p, cells):
    Nx, Ny = int(p.Nx), int(p.Ny)
    return cells % Nx, (cells // Nx) % Ny, cells // (Nx * Ny)


def ddf_locations(p, cells, t):
    """int64 [19, K]: the image elements cell n loads at parity t&1. f[i] (i odd) comes from its own slot i (odd t) / i+1 (even t), f[i+1] from slot i+1 / i of
    the neighbour n + c_i; store_f writes f[i] where f[i+1] was loaded and f[i+1] where f[i] was (so every element belongs to exactly one cell)."""
    Nx, Ny, Nz = int(p.Nx), int(p.Ny), int(p.Nz)
    N = Nx * Ny * Nz
    cells = np.asarray(cells, np.int64)
    x, y, z = _coords(p, cells)
    odd = int(t) & 1
    loc = np.empty((19, cells.size), np.int64)
    loc[0] = cells
    for i in range(1, 19, 2):
        j = (x + CX[i]) % Nx + ((y + CY[i]) % Ny + ((z + CZ[i]) % Nz) * Ny) * Nx
        loc[i] = (i if odd else i + 1) * N + cells
        loc[i + 1] = (i + 1 if odd else i) * N + j
    return loc


def store_locations(loc):
    """[19, K]: where the post-collision f[i] goes -- the element f[i+1] was loaded from, and vice versa."""
    out = np.empty_like(loc)
    out[0] = loc[0]
    out[1::2], out[2::2] = loc[2::2], loc[1::2]
    return out


def executes(p, flags):
    """int64 cells the step runs (FX/kernel.cpp:1478-1482): owned (not a halo layer of a decomposed axis), not TYPE_S, not TYPE_G."""
    flags = np.asarray(flags, np.uint8)
    cells = np.arange(flags.size, dtype=np.int64)
    x, y, z = _coords(p, cells)
    halo = np.zeros(flags.size, bool)
    for D, c, n in ((p.Dx, x, p.Nx), (p.Dy, y, p.Ny), (p.Dz, z, p.Nz)):
        if D > 1:
            halo |= (c == 0) | (c >= n - 1)
    run = ~halo & ((flags & TYPE_BO) != TYPE_S) & ((flags & TYPE_SU) != TYPE_G)
    return cells[run]


def f_eq(rho, ux, uy, uz, rhom1=None):
    """float64 [19, K]: w_i (rho (1 + 3 c.u + 9/2 (c.u)^2 - 3/2 u^2) - 1), i.e. w_i rho (...) + w_i (rho - 1) with `rhom1` standing for rho - 1."""
    rhom1 = rho - 1.0 if rhom1 is None else rhom1
    cu = CX[:, None] * ux + CY[:, None] * uy + CZ[:, None] * uz
    return W[:, None] * (rho * (3.0 * cu + 4.5 * cu * cu - 1.5 * (ux * ux + uy * uy + uz * uz)) + rhom1)


def _moments(f):
    rho = f.sum(0) + 1.0
    return rho, (CX @ f) / rho, (CY @ f) / rho, (CZ @ f) / rho


def _frame(p):
    Dx, Dy, Dz = int(p.Dx), int(p.Dy), int(p.Dz)
    Nxg, Nyg, Nzg = (int(p.Nx) - 2 * (Dx > 1)) * Dx, (int(p.Ny) - 2 * (Dy > 1)) * Dy, (int(p.Nz) - 2 * (Dz > 1)) * Dz
    return Nxg, Nyg, Nzg


def body_force(p, cells, bo, u, rho, ux, uy, uz, f, omega, zones):
    """Global force + Coriolis, plus buffer nudging and the top sponge (`zones`; not on TYPE_E cells) -- luw_force of the C oracle, sin^2 ramps in double."""
    N = int(p.Nx) * int(p.Ny) * int(p.Nz)
    fx, fy, fz = (F64(F32(v)) for v in f)
    ox, oy, oz = (F64(F32(v)) for v in omega)
    Fx = fx - 2.0 * rho * (oy * uz - oz * uy)
    Fy = fy - 2.0 * rho * (oz * ux - ox * uz)
    Fz = fz - 2.0 * rho * (ox * uy - oy * ux)
    if not zones:
        return Fx, Fy, Fz
    Nxg, Nyg, Nzg = _frame(p)
    Nx, Ny, Nz = int(p.Nx), int(p.Ny), int(p.Nz)
    Ox, Oy, Oz = int(p.Ox), int(p.Oy), int(p.Oz)
    wx, ex, sy, ny, tz = -Ox, Nxg - 1 - Ox, -Oy, Nyg - 1 - Oy, Nzg - 1 - Oz
    has_w, has_e, has_s, has_n, has_t = 0 <= wx < Nx, 0 <= ex < Nx, 0 <= sy < Ny, 0 <= ny < Ny, 0 <= tz < Nz
    x, y, z = _coords(p, cells)
    live = bo != TYPE_E
    if p.features & BUFFER_NUDGING:
        Nb = int(p.buffer_N)
        xg, yg, zg = x + Ox, y + Oy, z + Oz
        dw, de, ds, dn, dt = xg, Nxg - 1 - xg, yg, Nyg - 1 - yg, Nzg - 1 - zg
        face = int(p.downstream_face)
        dmin = np.full(cells.size, Nb + 1, np.int64)
        nref = cells.copy()
        for inside, d, ref in ((face != 1 and has_w, dw, wx + (y + z * Ny) * Nx), (face != 2 and has_e, de, ex + (y + z * Ny) * Nx),
                               (face != 3 and has_s, ds, x + (sy + z * Ny) * Nx), (face != 4 and has_n, dn, x + (ny + z * Ny) * Nx),
                               (has_t, dt, x + (y + tz * Ny) * Nx)):
            if inside:
                take = (d >= 0) & (d <= Nb) & (d < dmin)
                dmin = np.where(take, d, dmin)
                nref = np.where(take, ref, nref)
        act = live & (dmin <= Nb)
        wb = np.sin(HALF_PI * (1.0 - dmin / Nb)) ** 2 * F64(F32(p.buffer_inv_tau))
        wb = np.where(act, wb, 0.0)
        Fx = Fx + rho * (wb * (u[nref] - ux))
        Fy = Fy + rho * (wb * (u[N + nref] - uy))
        if int(p.buffer_nudge_vertical) == 1:
            Fz = Fz + rho * (wb * (u[2 * N + nref] - uz))
    if (p.features & TOP_SPONGE) and has_t:
        Ns = int(p.sponge_N)
        dt = (Nzg - 2) - (z + Oz)
        act = live & (dt >= 0) & (dt < Ns)
        xi = 1.0 - dt / (Ns - 1) if Ns > 1 else np.ones(cells.size)
        sigma = np.where(act, F64(F32(p.sponge_inv_tau)) * np.sin(HALF_PI * xi) ** 2, 0.0)
        nref = x + (y + tz * Ny) * Nx
        Fx = Fx + rho * sigma * (u[nref] - ux)
        Fy = Fy + rho * sigma * (u[N + nref] - uy)
        Fz = Fz + rho * sigma * (u[2 * N + nref] - uz)
    return Fx, Fy, Fz


def stream_collide(fi, flags, rho, u, p, t, f=(0.0, 0.0, 0.0), omega=(0.0, 0.0, 0.0), defect=None):
    """One step. `defect` (bar-separation tests only) injects a known bug: "no_forcing" (Guo term dropped, the force half-step kept) or "partner_rhom1"
    (a non-TYPE_E cell whose x pair partner -- cells 2k, 2k+1 of a row -- is TYPE_E uses the partner's boundary rho - 1 in its equilibrium)."""
    fi = np.asarray(fi, F64)
    flags = np.asarray(flags, np.uint8)
    N = flags.size
    feat = int(p.features)
    cells = executes(p, flags)
    loc = ddf_locations(p, cells, t)
    fin = fi[loc]
    bo = flags[cells] & TYPE_BO
    is_e = (bo == TYPE_E) if feat & EQUILIBRIUM_BOUNDARIES else np.zeros(cells.size, bool)
    r, ux, uy, uz = _moments(fin)
    r = np.where(is_e, rho[cells], r)
    ux, uy, uz = (np.where(is_e, u[c * N + cells], v) for c, v in enumerate((ux, uy, uz)))
    Fx, Fy, Fz = body_force(p, cells, bo, u, r, ux, uy, uz, f, omega, zones=True)
    if feat & VOLUME_FORCE:
        ux, uy, uz = (np.clip(v + F * (0.5 / r), -LAT_C, LAT_C) for v, F in ((ux, Fx), (uy, Fy), (uz, Fz)))
        uF = -THIRD * (ux * Fx + uy * Fy + uz * Fz)
        cF = CX[:, None] * Fx + CY[:, None] * Fy + CZ[:, None] * Fz
        cu = CX[:, None] * ux + CY[:, None] * uy + CZ[:, None] * uz
        Fin = 9.0 * W[:, None] * np.where(np.arange(19)[:, None] == 0, uF, cF * (cu + THIRD) + uF)
    else:
        ux, uy, uz = (np.clip(v, -LAT_C, LAT_C) for v in (ux, uy, uz))
        Fin = np.zeros_like(fin)
    rho_out, u_out = np.array(rho, F64), np.array(u, F64)
    if feat & UPDATE_FIELDS:
        wr = cells[~is_e]
        rho_out[wr] = r[~is_e]
        for c, v in enumerate((ux, uy, uz)):
            u_out[c * N + wr] = v[~is_e]
    rhom1 = r - 1.0
    if defect == "partner_rhom1":
        x = cells % int(p.Nx)
        partner = np.where(x % 2 == 0, cells + 1, cells - 1)
        ok = (partner // int(p.Nx) == cells // int(p.Nx)) & (partner < N)
        partner = np.where(ok, partner, cells)
        take = ok & ~is_e & ((flags[partner] & TYPE_BO) == TYPE_E) & bool(feat & EQUILIBRIUM_BOUNDARIES)
        rhom1 = np.where(take, np.asarray(rho, F64)[partner] - 1.0, rhom1)
    feq = f_eq(r, ux, uy, uz, rhom1)
    w = np.full(cells.size, F64(F32(p.w)))
    if feat & SUBGRID:
        tau0 = 1.0 / w
        neq = fin[1:] - feq[1:]
        cx, cy, cz = CX[1:, None], CY[1:, None], CZ[1:, None]
        Hxx, Hyy, Hzz = (cx * cx * neq).sum(0), (cy * cy * neq).sum(0), (cz * cz * neq).sum(0)
        Hxy, Hxz, Hyz = (cx * cy * neq).sum(0), (cx * cz * neq).sum(0), (cy * cz * neq).sum(0)
        Qn = Hxx * Hxx + Hyy * Hyy + Hzz * Hzz + 2.0 * (Hxy * Hxy + Hxz * Hxz + Hyz * Hyz)
        w = 2.0 / (tau0 + np.sqrt(tau0 * tau0 + SMAG * np.sqrt(Qn) / r))
    if feat & VOLUME_FORCE and defect != "no_forcing":
        Fin = Fin * (1.0 - 0.5 * w)
    elif defect == "no_forcing":
        Fin = np.zeros_like(fin)
    fout = np.where(is_e, feq, (1.0 - w) * fin + w * feq + Fin)
    out = fi.copy()
    sto = store_locations(loc)
    out[sto] = fout
    written = np.zeros(fi.size, bool)
    written[sto] = True
    scale = np.zeros(fi.size, F64)
    scale[sto] = np.abs(fin) + np.abs(feq) + W[:, None]
    return Step(out, rho_out, u_out, written, scale)


def update_fields(fi, flags, rho, u, p, t, f=(0.0, 0.0, 0.0), omega=(0.0, 0.0, 0.0)):
    """(rho, u) after the update_fields kernel at parity t&1: moments of the streamed-in DDFs, force half-step (no relaxation zones) and clamp; TYPE_E cells
    keep their boundary values when EQUILIBRIUM_BOUNDARIES is on."""
    fi = np.asarray(fi, F64)
    flags = np.asarray(flags, np.uint8)
    N = flags.size
    feat = int(p.features)
    cells = executes(p, flags)
    fin = fi[ddf_locations(p, cells, t)]
    bo = flags[cells] & TYPE_BO
    r, ux, uy, uz = _moments(fin)
    if feat & VOLUME_FORCE:
        Fx, Fy, Fz = body_force(p, cells, bo, u, r, ux, uy, uz, f, omega, zones=False)
        ux, uy, uz = (v + F * (0.5 / r) for v, F in ((ux, Fx), (uy, Fy), (uz, Fz)))
    ux, uy, uz = (np.clip(v, -LAT_C, LAT_C) for v in (ux, uy, uz))
    keep = (bo == TYPE_E) if feat & EQUILIBRIUM_BOUNDARIES else np.zeros(cells.size, bool)
    rho_out, u_out = np.array(rho, F64), np.array(u, F64)
    wr = cells[~keep]
    rho_out[wr] = r[~keep]
    for c, v in enumerate((ux, uy, uz)):
        u_out[c * N + wr] = v[~keep]
    return rho_out, u_out
