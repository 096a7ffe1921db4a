"""TEST INFRASTRUCTURE: numpy float32 restatement of the pedestrian-level wind statistics (csrc/lbm_wind_stats.cuh, luw_wind_stats_*, lbm.WindStatistics).
Only tests/ may import this; the product path never does. numpy rounds every elementwise float32 operation separately (no FMA) and np.sqrt is correctly rounded,
which is what the kernel's __fmul_rn / __fadd_rn / __fsqrt_rn do.

  column_ground    k_column_ground over a flags image
  layer_cells      the per-height cell lists of lbm.wind_layer_cells (global lattice, one domain)
  WindStatsOracle  k_wind_stats_accumulate
"""
import numpy as np

F32 = np.float32
NONE = np.uint32(0xFFFFFFFF)
PAIRS = ((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))  # uu vv ww uv uw vw


def column_ground(flags, Nx, Ny, Nz, z0=0, z1=None, Oz=0):
    """uint32 [Ny, Nx]: Oz + z of the lowest cell z0 <= z < z1 of each column with (flags & 0x03) != 0x01, 0xFFFFFFFF if none."""
    z1 = Nz if z1 is None else z1
    f = np.asarray(flags, np.uint8).reshape(Nz, Ny, Nx)[z0:z1]
    open_ = (f & 0x03) != 0x01
    first = np.argmax(open_, axis=0)
    return np.where(open_.any(axis=0), (first + z0 + Oz).astype(np.uint32), NONE).astype(np.uint32)


def layer_cells(flags, Nx, Ny, Nz, ground, heights):
    """Per height h_k: the cells at z = ground + h_k that lie inside the lattice and are plain fluid ((flags & 0x03) == 0), in (y, x) order.
    Returns (dense cell indices, slots k*Nx*Ny + y*Nx + x)."""
    f = np.asarray(flags, np.uint8)
    cells, slots = [], []
    for k, h in enumerate(heights):
        for y in range(Ny):
            for x in range(Nx):
                g = int(ground[y, x])
                if g == 0xFFFFFFFF or g + h >= Nz:
                    continue
                n = x + (y + (g + h) * Ny) * Nx
                if f[n] & 0x03 == 0:
                    cells.append(n)
                    slots.append(k * Nx * Ny + y * Nx + x)
    return np.array(cells, np.uint64), np.array(slots, np.int64)


class WindStatsOracle:
    """Accumulators of `count` cells, SoA like the device: mean (3, count), C (6, count), mean_s, m2_s, max_s, exceed (thresholds, count)."""

    def __init__(self, count, thresholds=()):
        self.thresholds = np.asarray(thresholds, F32)
        self.mean = np.zeros((3, count), F32)
        self.C = np.zeros((6, count), F32)
        self.mean_s, self.m2_s, self.max_s = np.zeros(count, F32), np.zeros(count, F32), np.zeros(count, F32)
        self.exceed = np.zeros((self.thresholds.size, count), np.uint32)
        self.n = 0

    def accumulate(self, ux, uy, uz):
        self.n += 1
        inv_n = F32(1.0) / F32(self.n)
        x = [np.asarray(v, F32) for v in (ux, uy, uz)]
        d, e = [], []
        for c in range(3):
            d.append(x[c] - self.mean[c])
            self.mean[c] = self.mean[c] + d[c] * inv_n
            e.append(x[c] - self.mean[c])
        for j, (a, b) in enumerate(PAIRS):
            self.C[j] = self.C[j] + d[a] * e[b]
        s = np.sqrt((x[0] * x[0] + x[1] * x[1]) + x[2] * x[2])
        ds = s - self.mean_s
        self.mean_s = self.mean_s + ds * inv_n
        self.m2_s = self.m2_s + ds * (s - self.mean_s)
        self.max_s = np.fmax(self.max_s, s)
        for j, t in enumerate(self.thresholds):
            self.exceed[j] += (s > t).astype(np.uint32)
