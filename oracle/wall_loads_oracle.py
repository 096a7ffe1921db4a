"""TEST INFRASTRUCTURE: numpy restatement of the wind loads on buildings (csrc/lbm_wall_loads.cuh, luw_solid_surface, luw_wall_loads_*, lbm.WallLoads,
LBM_WallLoads). Only tests/ may import this; the product path never does. numpy rounds every elementwise float32 / float64 operation separately (no FMA),
which is what the kernels' __fadd_rn / __fsub_rn / __fmul_rn / __dadd_rn / __dsub_rn / __dmul_rn do.

  surface           listed cells and their counted links over a flags image (one domain = the global lattice)
  load_f            the DDFs load_f<P> reads at a cell, from a dense DDF image (decoded with the oracle's codecs)
  cell_forces       F = 2 m per cell, float32, the momentum sums of rho_u left to right with non-counted links as +0.0
  moments           M = (r - r0) x F per cell, float64
  label_sums        the three-level per-label sum of the kernels (chunks of CHUNK cells, groups of GROUP chunks, then the groups; all within one label)
  WelfordF          the per-cell mean / M2 of F, float32
  footprint_labels  building columns grouped into 4-connected footprints, numbered in row-major order of first appearance (breadth-first flood fill)
  ref_points        the default reference point per label: the footprint's column-centre centroid at z = ground_z + 0.5, the origin for label 0
"""
from collections import deque

import numpy as np

F32, F64 = np.float32, np.float64
CHUNK = 32  # cells per first-level sum (WALL_CHUNK)
GROUP = 32  # first-level sums per second-level sum (WALL_GROUP)
NONE = 0xFFFFFFFF
# c_i in the DDF order of the kernels (lbm_common.cuh neighbors(): j[i] = n + c_i)
CX = np.array([0, 1, -1, 0, 0, 0, 0, 1, -1, 1, -1, 0, 0, 1, -1, 1, -1, 0, 0])
CY = np.array([0, 0, 0, 1, -1, 0, 0, 1, -1, 0, 0, 1, -1, -1, 1, 0, 0, 1, -1])
CZ = np.array([0, 0, 0, 0, 0, 1, -1, 0, 0, 1, -1, 1, -1, 0, 0, -1, 1, -1, 1])
# momentum sums of rho_u (lbm_common.cuh), left to right: (sign, DDF index)
MX = ((1, 1), (-1, 2), (1, 7), (-1, 8), (1, 9), (-1, 10), (1, 13), (-1, 14), (1, 15), (-1, 16))
MY = ((1, 3), (-1, 4), (1, 7), (-1, 8), (1, 11), (-1, 12), (1, 14), (-1, 13), (1, 17), (-1, 18))
MZ = ((1, 5), (-1, 6), (1, 9), (-1, 10), (1, 11), (-1, 12), (1, 16), (-1, 15), (1, 18), (-1, 17))


def _coords(cells, shape):
    Nx, Ny, _ = shape
    cells = np.asarray(cells, np.int64)
    return cells % Nx, (cells // Nx) % Ny, cells // (Nx * Ny)


def links(flags, shape, periodic, cells):
    """uint32 per cell: bit i set when the link of DDF i counts -- the partner n - c_i is not solid and is reached without crossing a face of a non-periodic axis."""
    Nx, Ny, Nz = shape
    f = np.asarray(flags, np.uint8).reshape(Nz, Ny, Nx)
    x, y, z = _coords(cells, shape)
    m = np.zeros(x.size, np.uint32)
    for i in range(1, 19):
        px, py, pz = x - CX[i], y - CY[i], z - CZ[i]
        inside = np.ones(x.size, bool)
        for a, (p, n) in enumerate(((px, Nx), (py, Ny), (pz, Nz))):
            if not periodic[a]:
                inside &= (p >= 0) & (p < n)
        solid = (f[pz % Nz, py % Ny, px % Nx] & 0x03) == 0x01
        m |= np.where(inside & ~solid, np.uint32(1 << i), np.uint32(0))
    return m


def surface(flags, shape, periodic=(False, False, False)):
    """(listed cells ascending, their link masks): solid cells ((flags & 0x03) == 0x01) with at least one counted link."""
    solid = np.nonzero((np.asarray(flags, np.uint8) & 0x03) == 0x01)[0]
    m = links(flags, shape, periodic, solid)
    keep = m != 0
    return solid[keep].astype(np.uint64), m[keep]


_TABLES = {}


def decode(fi, precision):
    """DDF storage -> float32 as the kernels' Ddf<P>::dec: FP16S = binary16 x 2^-15, FP16C = the 1-4-11 format (oracle codecs)."""
    if precision == 0:
        return np.asarray(fi, F32)
    if precision not in _TABLES:
        from oracle import oracle as O
        orc = O.Oracle()
        if precision == 1:
            t = np.array([orc.half_to_float(h) for h in range(65536)], F32) * F32(3.0517578e-05)
        else:
            t = np.array([orc.fp16c_to_float(h) for h in range(65536)], F32)
        _TABLES[precision] = t.astype(F32)
    return _TABLES[precision][np.asarray(fi, np.uint16)]


def load_f(fi, shape, precision, cells, odd):
    """float32 [19, K]: f[i] at the cells as load_f<P> reads them (Esoteric-Pull, time parity `odd`), from the dense image fi[i*N + n] (periodic wrap)."""
    Nx, Ny, Nz = shape
    N = Nx * Ny * Nz
    d = decode(fi, precision).reshape(19, N)
    x, y, z = _coords(cells, shape)
    n = np.asarray(cells, np.int64)
    f = np.empty((19, n.size), F32)
    f[0] = d[0, n]
    for i in range(1, 19, 2):
        ji = ((x + CX[i]) % Nx) + ((y + CY[i]) % Ny + ((z + CZ[i]) % Nz) * Ny) * Nx
        f[i] = d[i if odd else i + 1, n]
        f[i + 1] = d[i + 1 if odd else i, ji]
    return f


def cell_forces(f, m):
    """float32 [3, K]: F = 2 m, the momentum sums evaluated left to right in float32 with the term of a non-counted link replaced by +0.0."""
    g = np.where(((np.asarray(m, np.uint32)[None, :] >> np.arange(19, dtype=np.uint32)[:, None]) & 1) == 1, f, F32(0.0)).astype(F32)
    out = []
    for terms in (MX, MY, MZ):
        s = g[terms[0][1]].copy()
        for sign, i in terms[1:]:
            s = (s + g[i]) if sign > 0 else (s - g[i])
        out.append(F32(2.0) * s)
    return np.array(out, F32)


def moments(F, gx, gy, gz, r0):
    """float64 [3, K]: (r - r0) x F, r the global integer coordinates, r0 [K, 3] per cell; products and differences rounded separately."""
    fx, fy, fz = (np.asarray(v, F32).astype(F64) for v in F)
    r0 = np.asarray(r0, F64)
    dx, dy, dz = np.asarray(gx, F64) - r0[:, 0], np.asarray(gy, F64) - r0[:, 1], np.asarray(gz, F64) - r0[:, 2]
    return np.array([dy * fz - dz * fy, dz * fx - dx * fz, dx * fy - dy * fx], F64)


def label_sums(F, M, labels, L, chunk=CHUNK, group=GROUP):
    """float64 [L, 6] (Fx Fy Fz Mx My Mz) in the kernels' order. The list is sorted by label; each label's cells are cut into chunks of `chunk` from its first
    cell, every chunk summed in index order from +0.0; the label's chunk sums are cut into groups of `group`, each summed in order from +0.0; then the label's
    group sums are added in order from +0.0."""
    labels = np.asarray(labels, np.int64)
    V = np.concatenate([np.asarray(F, F32).astype(F64), np.asarray(M, F64)]) if labels.size else np.zeros((6, 0), F64)
    out = np.zeros((L, 6), F64)

    def ordered(rows):
        s = np.zeros(6, F64)
        for r in rows:
            s = s + r
        return s
    for l in range(L):
        idx = np.nonzero(labels == l)[0]
        chunks = [ordered(V[:, k] for k in idx[c0:c0 + chunk]) for c0 in range(0, idx.size, chunk)]
        groups = [ordered(chunks[g0:g0 + group]) for g0 in range(0, len(chunks), group)]
        out[l] = ordered(groups)
    return out


class WelfordF:
    """Per-cell mean / M2 of F (3, count), float32, rounded like k_wall_cells."""

    def __init__(self, count):
        self.mean, self.m2 = np.zeros((3, count), F32), np.zeros((3, count), F32)
        self.n = 0

    def accumulate(self, F):
        self.n += 1
        inv_n = F32(1.0) / F32(self.n)
        F = np.asarray(F, F32)
        d = F - self.mean
        self.mean = self.mean + d * inv_n
        self.m2 = self.m2 + d * (F - self.mean)


def column_ground(flags, shape):
    """uint32 [Ny, Nx]: z of the lowest non-solid cell of every column, 0xFFFFFFFF if none."""
    Nx, Ny, Nz = shape
    open_ = (np.asarray(flags, np.uint8).reshape(Nz, Ny, Nx) & 0x03) != 0x01
    return np.where(open_.any(0), np.argmax(open_, 0), NONE).astype(np.uint32)


def footprint_labels(ground, ground_z=0):
    """uint32 [Ny, Nx]: 0 outside buildings; building columns (ground above ground_z + 1, 0xFFFFFFFF included) grouped into 4-connected components (no wrap
    across the lattice edges) numbered 1..B in row-major (y, x) order of first appearance."""
    g = np.asarray(ground).astype(np.int64)
    b = g > ground_z + 1
    Ny, Nx = b.shape
    lab = np.zeros((Ny, Nx), np.uint32)
    nxt = 0
    for y in range(Ny):
        for x in range(Nx):
            if b[y, x] and lab[y, x] == 0:
                nxt += 1
                lab[y, x] = nxt
                q = deque([(y, x)])
                while q:
                    cy, cx = q.popleft()
                    for ny, nx in ((cy - 1, cx), (cy + 1, cx), (cy, cx - 1), (cy, cx + 1)):
                        if 0 <= ny < Ny and 0 <= nx < Nx and b[ny, nx] and lab[ny, nx] == 0:
                            lab[ny, nx] = nxt
                            q.append((ny, nx))
    return lab


def ref_points(column_labels, L, ground_z=0):
    """float64 [L, 3]: per label l >= 1 the mean of its columns' (x, y) (integer sums divided by the column count) and z = ground_z + 0.5; the origin for
    label 0 and for a label without columns."""
    lab = np.asarray(column_labels, np.int64)
    out = np.zeros((L, 3), F64)
    for l in range(1, L):
        ys, xs = np.nonzero(lab == l)
        if xs.size:
            out[l] = (F64(int(xs.sum())) / F64(xs.size), F64(int(ys.sum())) / F64(xs.size), F64(ground_z) + F64(0.5))
    return out


def cell_labels(gx, gy, gz, column_labels, ground_z=0):
    """uint32 label per listed cell: its column's label above ground_z, 0 (terrain) at or below it."""
    lab = np.asarray(column_labels)[np.asarray(gy, np.int64), np.asarray(gx, np.int64)].astype(np.uint32)
    return np.where(np.asarray(gz) > ground_z, lab, 0).astype(np.uint32)
