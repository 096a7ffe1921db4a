"""Host-side mirror of the reference's `LBM` object (FX/lbm.hpp:223-633, FX/lbm.cpp:1057-1312) over the C ABI.

    lbm = LBM((Nx, Ny, Nz), D=(Dx, Dy, Dz), nu=..., precision=..., features=...)
    lbm.flags[...] / lbm.u[...] / lbm.rho[...]      global host images, reference layout n = x + (y + z*Ny)*Nx, u = [ux | uy | uz]
    lbm.run(steps)                                   first call initialises (upload + `initialize` kernel + halo fill), then steps
    lbm.read_from_device()                           device -> global host images

Two drivers share the domain split and the step sequence of the reference (`do_time_step`: stream_collide on every domain, then
`communicate_fi` axis by axis x -> y -> z):
  * LBM             one process owns all Dx*Dy*Dz domains (any mix of devices; several domains may share one GPU, which is how
                    decomposed runs are tested on a single B200). Halo payloads move device-to-device.
  * DistributedLBM  one process per GPU (torch.distributed, NCCL): each rank owns ONE domain; halo payloads move with batched
                    isend/irecv over NVLink. This replaces the host-staged exchange of FX/lbm.cpp:1907-1935.
torch is used for device buffers, streams and the process group only; all LBM work is in the CUDA library behind the C ABI.
"""
import numpy as np

from . import _cabi as A
from . import cases
from .domain import CellSet, Domain, WindStats
from .domain import WallLoads as DomainWallLoads
from .domain import Probes as DomainProbes
from .domain import Particles as DomainParticles

AXES = (0, 1, 2)


def split(shape, D):
    """Domain split of FX/lbm.cpp:1057-1073: global N rounded down to multiples of D, local N/D + 2 halo layers on decomposed axes,
    offset O = d*N/D - H. Returns (global shape, local shape, list of (d, O))."""
    D = tuple(int(v) for v in D)
    Ng = tuple((int(n) // d) * d for n, d in zip(shape, D))
    H = tuple(1 if d > 1 else 0 for d in D)
    Nl = tuple(n // d + 2 * h for n, d, h in zip(Ng, D, H))
    doms = []
    for dz in range(D[2]):
        for dy in range(D[1]):
            for dx in range(D[0]):
                d = (dx, dy, dz)
                doms.append((d, tuple(d[a] * (Ng[a] // D[a]) - H[a] for a in AXES)))
    return Ng, Nl, doms


def _local_index(Ng, Nl, O):
    """Global linear indices of every local cell (periodic at the global edges), the stitching of FX/lbm.hpp:274-297."""
    idx = [np.mod(np.arange(Nl[a]) + O[a], Ng[a]) for a in AXES]
    g = idx[0][None, None, :] + Ng[0] * (idx[1][None, :, None] + Ng[1] * idx[2][:, None, None])
    return g.reshape(-1)


class _Base:
    def __init__(self, shape, D=(1, 1, 1), nu=1.0 / 6.0, precision=A.FP32, features=A.UPDATE_FIELDS, arith=A.ARITH_FAST,
                 f=(0.0, 0.0, 0.0), omega=(0.0, 0.0, 0.0), w=None, alpha=0.0, beta=0.0, T_avg=1.0, **zones):
        self.D = tuple(int(v) for v in D)
        self.Ng, self.Nl, self._split = split(shape, self.D)
        self.N = int(np.prod(self.Ng))
        self.precision, self.features, self.arith = precision, features, arith
        self.w = cases.relaxation_rate(nu) if w is None else w
        self.f, self.omega = tuple(f), tuple(omega)
        self.zones = zones
        # thermal D3Q7 extension (features & TEMPERATURE): LBM ctor arguments alpha (thermal diffusion coefficient) and beta (thermal expansion
        # coefficient), FX/lbm.cpp:1040-1047; def_w_T = 1/(2 alpha + 1/2) in float arithmetic like FX/lbm.cpp:750
        self.thermal = bool(features & A.TEMPERATURE)
        self.w_T = float(cases.kernel_literal(np.float32(1.0) / (np.float32(2.0) * np.float32(alpha) + np.float32(0.5))))
        self.beta, self.T_avg = float(cases.kernel_literal(beta)), float(cases.kernel_literal(T_avg))
        self.t = 0
        self.initialized = False

    def _make_domain(self, d, O, device):
        dom = Domain(*self.Nl, D=self.D, O=O, precision=self.precision, features=self.features, w=self.w, arith=self.arith,
                     device=device, **self.zones)
        dom.f, dom.omega = self.f, self.omega
        if self.thermal:
            dom.set_thermal(self.w_T, self.beta, self.T_avg)
        return dom

    def set_coriolis(self, ox, oy, oz):  # FX/lbm.hpp:496-498
        self.omega = (ox, oy, oz)
        for dom in self.domains:
            dom.omega = self.omega

    def get_N(self):
        return self.N

    def get_t(self):
        return self.t


class LBM(_Base):
    """All domains in one process (reference: `LBM` with `lbm_domain[d]`, FX/lbm.hpp:426)."""

    def __init__(self, shape, D=(1, 1, 1), devices=None, **kw):
        super().__init__(shape, D, **kw)
        ndev = max(A.device_count(), 1)
        self.devices = list(devices) if devices is not None else [i % ndev for i in range(len(self._split))]
        self.domains = [self._make_domain(d, O, dev) for (d, O), dev in zip(self._split, self.devices)]
        self.rho = np.ones(self.N, np.float32)
        self.u = np.zeros(3 * self.N, np.float32)
        self.flags = np.zeros(self.N, np.uint8)
        self.T = np.ones(self.N, np.float32) if self.thermal else None
        self._gidx = [_local_index(self.Ng, self.Nl, O) for _, O in self._split]

    # ---- host <-> device (Memory_Container::write_to_device / read_from_device, FX/lbm.hpp:406-423)
    def write_to_device(self):
        for dom, g in zip(self.domains, self._gidx):
            dom.rho[:] = self.rho[g]
            dom.flags[:] = self.flags[g]
            for c in range(3):
                dom.u[c * dom.N:(c + 1) * dom.N] = self.u[c * self.N + g]
            if self.thermal:
                dom.T[:] = self.T[g]
            dom.upload_all()

    def read_from_device(self):
        H = tuple(1 if d > 1 else 0 for d in self.D)
        for dom, g in zip(self.domains, self._gidx):
            dom.download_all()
            keep = np.ones(self.Nl[::-1], bool)
            if H[0]: keep[:, :, 0] = keep[:, :, -1] = False
            if H[1]: keep[:, 0, :] = keep[:, -1, :] = False
            if H[2]: keep[0, :, :] = keep[-1, :, :] = False
            k = keep.reshape(-1)
            self.rho[g[k]] = dom.rho[k]
            self.flags[g[k]] = dom.flags[k]
            for c in range(3):
                self.u[c * self.N + g[k]] = dom.u[c * dom.N:(c + 1) * dom.N][k]
            if self.thermal:
                self.T[g[k]] = dom.T[k]

    # ---- halo exchange (FX/lbm.cpp:1895-1958): extract, peer copies and insert are enqueued by the library, stream-ordered
    def _handles(self):
        import ctypes as C
        if not hasattr(self, "_harr"):
            self._harr = (C.c_void_p * len(self.domains))(*[dom._h for dom in self.domains])
        return self._harr

    def communicate(self, payload):
        t = self.domains[0].t
        for axis in AXES:
            A.check(A.lib().luw_halo_exchange(self._handles(), len(self.domains), payload, axis, t))

    # ---- LBM::initialize / do_time_step / run (FX/lbm.cpp:1221-1312)
    def initialize(self):
        self.write_to_device()
        for dom in self.domains:
            dom.t = 1
        self.communicate(A.HALO_RHO_U_FLAGS)
        for dom in self.domains:
            dom.enqueue_initialize()
        self.communicate(A.HALO_RHO_U_FLAGS)
        self.communicate(A.HALO_FI)
        if self.thermal:  # communicate_T(); communicate_gi(): FX/lbm.cpp LBM::initialize
            self.communicate(A.HALO_T)
            self.communicate(A.HALO_GI)
        for dom in self.domains:
            dom.finish_queue()
            dom.t = 0
        self.t = 0
        self.initialized = True

    def do_time_step(self):
        for dom in self.domains:
            dom.f, dom.omega = self.f, self.omega
            dom.enqueue_stream_collide()
        self.communicate(A.HALO_FI)
        if self.thermal:
            self.communicate(A.HALO_GI)
        for dom in self.domains:
            dom.increment_time_step()
        self.t += 1

    def run(self, steps=1):
        if not self.initialized:
            self.initialize()
        if len(self.domains) == 1:
            dom = self.domains[0]
            dom.f, dom.omega = self.f, self.omega
            dom.run_steps(steps)
            self.t += steps
        else:
            A.check(A.lib().luw_run_steps_multi(self._handles(), len(self.domains), self.t, steps, *map(float, self.f), *map(float, self.omega)))
            for dom in self.domains:
                dom.increment_time_step(steps)
            self.t += steps
        for dom in self.domains:
            dom.finish_queue()

    def update_fields(self):
        for dom in self.domains:
            dom.enqueue_update_fields()

    def close(self):
        for dom in self.domains:
            dom.close()


def wind_layer_cells(dom, O, Ng, D, ground, heights):
    """The cells of one domain that pedestrian-level statistics cover: for every height h_k (cells), the OWNED cells at global z = ground + h_k whose flags are
    plain fluid ((flags & 0x03) == 0: no TYPE_S, no TYPE_E); cells above the lattice are left out. ground: uint32 [Ng_y, Ng_x], global z of the lowest non-solid
    cell per global column (0xFFFFFFFF: none). The flags are gathered from the device at the candidate cells (a cell set), so no host mirror is touched.
    Returns (local dense cell indices, slots), slots[i] = k*Ng_x*Ng_y + y*Ng_x + x of the global layer-major arrays, in that order."""
    H = tuple(1 if d > 1 else 0 for d in D)
    xs, ys = np.arange(H[0], dom.Nx - H[0]), np.arange(H[1], dom.Ny - H[1])
    gx, gy = xs + O[0], ys + O[1]  # owned cells never wrap
    g = ground[np.ix_(gy, gx)].astype(np.int64)
    cells, slots = [], []
    for k, h in enumerate(heights):
        zg = g + int(h)
        lz = zg - O[2]
        yy, xx = np.nonzero((g != 0xFFFFFFFF) & (zg < Ng[2]) & (lz >= H[2]) & (lz < dom.Nz - H[2]))
        cells.append(xs[xx] + (ys[yy] + lz[yy, xx] * dom.Ny) * dom.Nx)
        slots.append(k * Ng[0] * Ng[1] + gy[yy] * Ng[0] + gx[xx])
    cells, slots = np.concatenate(cells).astype(np.uint64), np.concatenate(slots).astype(np.int64)
    fl = np.zeros(cells.size, np.uint8)
    if cells.size:
        cs = CellSet(dom, cells)
        cs.download(A.FIELD_FLAGS, fl)
        dom.finish_queue()
        cs.close()
    keep = (fl & 0x03) == 0
    return cells[keep], slots[keep]


def global_column_ground(lbm):
    """uint32 [Ng_y, Ng_x]: global z of the lowest non-solid cell of every global column over the domains stacked in z (luw_column_ground per domain, minimum
    per column), 0xFFFFFFFF where there is none."""
    Ng = lbm.Ng
    H = tuple(1 if d > 1 else 0 for d in lbm.D)
    ground = np.full((Ng[1], Ng[0]), 0xFFFFFFFF, np.uint32)
    for dom, (_, O) in zip(lbm.domains, lbm._split):
        g = dom.column_ground()[H[1]:dom.Ny - H[1], H[0]:dom.Nx - H[0]]
        view = ground[O[1] + H[1]:O[1] + H[1] + g.shape[0], O[0] + H[0]:O[0] + H[0] + g.shape[1]]
        np.minimum(view, g, out=view)
    return ground


class WindStatistics:
    """Pedestrian-level wind statistics of an in-process `LBM` (all domains in this process) on surface-following layers: for every height h_k (cells) above the
    local ground or roof, the running mean and co-moments of u, mean / M2 / peak of the speed and threshold exceedance counts, accumulated on the device per sample
    (luw_wind_stats_*). Build it after the flags are on the device (after run(0) / initialize()).

    The ground of a global column is the lowest non-solid cell over the domains stacked in z (luw_column_ground per domain, minimum per column); each domain then
    lists its owned plain-fluid cells at ground + h_k. The one-process-per-GPU DistributedLBM is not covered here; the C ABI allows the same construction there:
    per-rank luw_column_ground, a min-reduce over the ranks stacked in z, then per-rank lists."""

    def __init__(self, lbm, heights, thresholds=()):
        self.lbm = lbm
        self.heights = [int(h) for h in heights]
        self.thresholds = np.ascontiguousarray(thresholds, np.float32)
        Ng = lbm.Ng
        self.ground = global_column_ground(lbm)
        self._stats, self._slots = [], []
        for dom, (_, O) in zip(lbm.domains, lbm._split):
            cells, slots = wind_layer_cells(dom, O, Ng, lbm.D, self.ground, self.heights)
            self._stats.append(WindStats(dom, cells, self.thresholds))
            self._slots.append(slots)

    def accumulate(self):
        if not self.lbm.features & A.UPDATE_FIELDS:  # rho / u are not stored every step
            self.lbm.update_fields()
        for st in self._stats:
            st.accumulate()

    def reset(self):
        for st in self._stats:
            st.reset()

    def download(self):
        """-> dict of global layer-major arrays [..., k, y, x]: mean_u (3, K, Ny, Nx), comoment (6, ...: uu vv ww uv uw vw), mean_speed, m2_speed, max_speed,
        exceed (thresholds, ...), valid (bool: the slot is a listed cell; float fields are NaN and counters 0 elsewhere) and the sample count."""
        Ng, K, T = self.lbm.Ng, len(self.heights), int(self.thresholds.size)
        M = K * Ng[1] * Ng[0]
        out = {"mean_u": np.full((3, M), np.nan, np.float32), "comoment": np.full((6, M), np.nan, np.float32), "mean_speed": np.full(M, np.nan, np.float32),
               "m2_speed": np.full(M, np.nan, np.float32), "max_speed": np.full(M, np.nan, np.float32), "exceed": np.zeros((T, M), np.uint32),
               "valid": np.zeros(M, bool)}
        samples = 0
        for st, slots in zip(self._stats, self._slots):
            mean_u, com, ms, m2, mx, ex, samples = st.download()
            out["mean_u"][:, slots], out["comoment"][:, slots], out["exceed"][:, slots] = mean_u, com, ex
            out["mean_speed"][slots], out["m2_speed"][slots], out["max_speed"][slots] = ms, m2, mx
            out["valid"][slots] = True
        out = {k: v.reshape(v.shape[:-1] + (K, Ng[1], Ng[0])) for k, v in out.items()}
        out["samples"] = samples
        return out

    def close(self):
        for st in self._stats:
            st.close()


def footprint_labels(ground, ground_z=0):
    """uint32 [Ny, Nx] from the global column ground: 0 outside buildings; a building column is one whose ground (lowest non-solid z) lies above ground_z + 1
    (an all-solid column included). Building columns are grouped into 4-connected footprints (no wrap across the lattice edges), numbered 1..B in row-major
    (y, x) order of first appearance. Minimum-index propagation with pointer jumping: every column ends with the smallest raster index of its footprint."""
    b = np.asarray(ground).astype(np.int64) > int(ground_z) + 1
    Ny, Nx = b.shape
    big = Ny * Nx
    lab = np.where(b, np.arange(big, dtype=np.int64).reshape(Ny, Nx), big)
    while True:
        n = lab.copy()
        np.minimum(n[1:], lab[:-1], out=n[1:])
        np.minimum(n[:-1], lab[1:], out=n[:-1])
        np.minimum(n[:, 1:], lab[:, :-1], out=n[:, 1:])
        np.minimum(n[:, :-1], lab[:, 1:], out=n[:, :-1])
        n = np.where(b, n, big)
        n = np.where(b, n.reshape(-1)[np.minimum(n, big - 1)], big)  # pointer jumping: the label of the column one points at
        if np.array_equal(n, lab):
            break
        lab = n
    out = np.zeros((Ny, Nx), np.uint32)
    roots = np.unique(lab[b])  # ascending smallest raster index = order of first appearance
    out[b] = (np.searchsorted(roots, lab[b]) + 1).astype(np.uint32)
    return out


def footprint_ref_points(column_labels, label_count, ground_z=0):
    """float64 [L, 3]: per label l >= 1 the centroid of its columns' centres (x, y) -- integer sums divided by the column count -- at z = ground_z + 0.5, the
    base of the building, so that the moment is the overturning moment; the origin for label 0 (terrain) and for a label without columns."""
    lab = np.asarray(column_labels).astype(np.int64).reshape(-1)
    Ny, Nx = np.asarray(column_labels).shape
    xs, ys = np.tile(np.arange(Nx, dtype=np.int64), Ny), np.repeat(np.arange(Ny, dtype=np.int64), Nx)
    cnt = np.bincount(lab, minlength=label_count)[:label_count]
    sx, sy = np.bincount(lab, xs, label_count)[:label_count], np.bincount(lab, ys, label_count)[:label_count]
    out = np.zeros((label_count, 3), np.float64)
    has = cnt > 0
    has[0] = False
    out[has, 0], out[has, 1] = sx[has] / cnt[has], sy[has] / cnt[has]
    out[has, 2] = float(ground_z) + 0.5
    return out


class WallLoads:
    """Wind loads on the buildings of an in-process `LBM` (all domains in this process): per sample and label (building) the momentum-exchange force and its
    moment about the label's reference point, and per surface cell the running mean / M2 of the force (luw_solid_surface, luw_wall_loads_*). Build it after
    the flags are on the device (after run(0) / initialize()).

    Every domain lists its solid cells that touch the fluid (luw_solid_surface; `periodic` per axis: links across a global face of a non-periodic axis do not
    count). Labels: by default from the global column ground (as in WindStatistics) -- footprint_labels(ground, ground_z) -- or from `column_labels[Ny][Nx]`
    (for example building ids from GIS data); a listed cell takes its column's label above z = ground_z and 0 (terrain) at or below it. Reference points:
    `ref_points[L][3]` or footprint_ref_points (the footprint's centroid at its base; the origin for label 0).

    accumulate() samples the current state without update_fields; the samples stay on the device until `capacity` of them are pending, then they are drained
    (the only host synchronisation). Forces and moments are in lattice units and gauge (relative to the reference pressure 1/3); dividing by 1/2 rho U^2 A for
    coefficients is the caller's business. The one-process-per-GPU DistributedLBM is not covered (it would need a cross-rank sum per sample)."""

    def __init__(self, lbm, ground_z=0, column_labels=None, ref_points=None, periodic=(False, False, False), capacity=256):
        self.lbm = lbm
        self.ground_z = int(ground_z)
        self.capacity = int(capacity)
        self.periodic_mask = sum(1 << a for a in AXES if periodic[a])
        Ng = lbm.Ng
        self.ground = global_column_ground(lbm)
        self.column_labels = footprint_labels(self.ground, self.ground_z) if column_labels is None else np.asarray(column_labels).astype(np.uint32).reshape(Ng[1], Ng[0])
        self.L = int(self.column_labels.max()) + 1
        self.ref_points = footprint_ref_points(self.column_labels, self.L, self.ground_z) if ref_points is None else \
            np.ascontiguousarray(ref_points, np.float64).reshape(self.L, 3)
        self._loads, self._global, self._labels = [], [], []
        for dom, (_, O) in zip(lbm.domains, lbm._split):
            local = dom.solid_surface(self.periodic_mask).astype(np.int64)
            gx, gy, gz = local % dom.Nx + O[0], (local // dom.Nx) % dom.Ny + O[1], local // (dom.Nx * dom.Ny) + O[2]  # owned cells never wrap
            lab = np.where(gz > self.ground_z, self.column_labels[gy, gx], 0).astype(np.uint32)
            order = np.lexsort((local, lab))
            self._loads.append(DomainWallLoads(dom, local[order], lab[order], self.L, self.ref_points, self.periodic_mask, self.capacity))
            self._global.append((gx + (gy + gz * Ng[1]) * Ng[0])[order])
            self._labels.append(lab[order])
        self._pending = 0
        self._series = []

    def accumulate(self):
        if self._pending == self.capacity:
            self._drain()
        for dom, st in zip(self.lbm.domains, self._loads):
            st.accumulate(dom.t)
        self._pending += 1

    def _drain(self):
        parts = [st.drain() for st in self._loads]
        total = parts[0].copy()
        for p in parts[1:]:  # domain order
            total += p
        if total.shape[0]:
            self._series.append(total)
        self._pending = 0

    def series(self):
        """-> float64 [samples, L, 6]: Fx Fy Fz Mx My Mz per sample and label since construction / reset, summed over the domains in domain order."""
        self._drain()
        return np.concatenate(self._series) if self._series else np.zeros((0, self.L, 6), np.float64)

    def summary(self):
        """-> dict of float64 [L, 6]: mean, std (population), min and max over the samples of the series, and the sample count."""
        s = self.series()
        if not s.shape[0]:
            raise ValueError("no samples accumulated")
        return {"mean": s.mean(0), "std": s.std(0), "min": s.min(0), "max": s.max(0), "samples": s.shape[0]}

    def surface(self):
        """-> dict over all listed cells, ascending global index n = x + (y + z*Ny)*Nx: cell, x, y, z, label, mean_F [3, K], m2_F [3, K], samples."""
        Ng = self.lbm.Ng
        cell = np.concatenate(self._global)
        label = np.concatenate(self._labels)
        mean, m2, samples = [], [], 0
        for st in self._loads:
            a, b, samples = st.download_cells()
            mean.append(a)
            m2.append(b)
        order = np.argsort(cell, kind="stable")
        cell = cell[order]
        return {"cell": cell.astype(np.uint64), "x": cell % Ng[0], "y": (cell // Ng[0]) % Ng[1], "z": cell // (Ng[0] * Ng[1]), "label": label[order],
                "mean_F": np.concatenate(mean, axis=1)[:, order], "m2_F": np.concatenate(m2, axis=1)[:, order], "samples": samples}

    def reset(self):
        for st in self._loads:
            st.reset()
        self._pending = 0
        self._series = []

    def close(self):
        for st in self._loads:
            st.close()


def probe_owners(Ng, D, split_offsets, Nl, points):
    """Which block owns each global point: -> (block [P], local dense index [P]). Halo layers are never owners, so every point of the lattice has exactly one.
    Raises ValueError for points outside the lattice [0, Ng)."""
    p = np.asarray(points, np.int64).reshape(-1, 3)
    if ((p < 0) | (p >= np.asarray(Ng, np.int64))).any():
        raise ValueError("probe points must lie inside the lattice [0, Ng)")
    H = np.array([1 if d > 1 else 0 for d in D], np.int64)
    Nl = np.asarray(Nl, np.int64)
    block, local = np.full(p.shape[0], -1, np.int64), np.zeros(p.shape[0], np.int64)
    for b, O in enumerate(split_offsets):
        q = p - np.asarray(O, np.int64)
        own = ((q >= H) & (q < Nl - H)).all(axis=1)
        block[own] = b
        local[own] = q[own, 0] + (q[own, 1] + q[own, 2] * Nl[1]) * Nl[0]
    assert (block >= 0).all()
    return block, local


def probe_columns(ground, xy, heights, Nz):
    """Vertical profiles that follow terrain and roofs: the points (x, y, ground + h) for every column (x, y) of `xy` [M, 2] and height h (cells) of `heights`,
    ground from global_column_ground (uint32 [Ny, Nx]). A column without ground (0xFFFFFFFF) or whose top point would lie at or above Nz is dropped.
    -> (points int64 [M_kept * len(heights), 3] ordered [column][height], dropped: indices into xy of the dropped columns)."""
    g = np.asarray(ground)
    xy = np.asarray(xy, np.int64).reshape(-1, 2)
    h = np.asarray(heights, np.int64).reshape(-1)
    if ((xy < 0) | (xy >= np.array([g.shape[1], g.shape[0]]))).any():
        raise ValueError("columns must lie inside the lattice")
    if (h < 0).any():
        raise ValueError("heights must be non-negative")
    G = g[xy[:, 1], xy[:, 0]].astype(np.int64)
    keep = (G != 0xFFFFFFFF) & (G + (h.max() if h.size else 0) < int(Nz))
    k = np.nonzero(keep)[0]
    pts = np.empty((k.size, h.size, 3), np.int64)
    pts[..., 0] = xy[k, 0, None]
    pts[..., 1] = xy[k, 1, None]
    pts[..., 2] = G[k, None] + h[None, :]
    return pts.reshape(-1, 3), np.nonzero(~keep)[0]


class Probes:
    """Time series of rho, u (and T on thermal lattices) at points of an in-process `LBM` (all domains in this process), sampled on the device without
    update_fields over the lattice (luw_probes_*). `points` [P, 3]: global lattice coordinates (ValueError outside the lattice); each goes to the one block
    that owns it. sample() takes the values update_fields + a read would give at the current time step; the samples stay on the device until `capacity`
    are pending, then they are drained (the only host synchronisation). Build it after initialisation (run(0)) when the domains do not store rho / u every
    step, as update_fields needs DDFs to read. The one-process-per-GPU DistributedLBM is not covered."""

    def __init__(self, lbm, points, capacity=256):
        self.lbm = lbm
        self.points = np.asarray(points, np.int64).reshape(-1, 3)
        self.P, self.capacity = self.points.shape[0], int(capacity)
        self.comps = 5 if lbm.thermal else 4
        block, local = probe_owners(lbm.Ng, lbm.D, [O for _, O in lbm._split], lbm.Nl, self.points)
        self._probes, self._slots = [], []
        for b, dom in enumerate(lbm.domains):
            slot = np.nonzero(block == b)[0]
            self._probes.append(DomainProbes(dom, local[slot], self.capacity))
            self._slots.append(slot)
        self._pending = 0
        self._t, self._series = [], []

    def sample(self):
        if self._pending == self.capacity:
            self._drain()
        for pr in self._probes:
            pr.sample()
        self._t.append(self.lbm.domains[0].t)
        self._pending += 1

    def _drain(self):
        out = np.empty((self._pending, self.comps, self.P), np.float32)
        for pr, slot in zip(self._probes, self._slots):
            out[:, :, slot] = pr.drain()
        if out.shape[0]:
            self._series.append(out)
        self._pending = 0

    def series(self):
        """-> dict: t int64 [S], rho float32 [S, P], u float32 [S, 3, P] (and T [S, P] on thermal lattices), points in the caller's order, since construction /
        reset."""
        self._drain()
        s = np.concatenate(self._series) if self._series else np.zeros((0, self.comps, self.P), np.float32)
        out = {"t": np.asarray(self._t, np.int64), "rho": s[:, 0].copy(), "u": s[:, 1:4].copy()}
        if self.comps == 5:
            out["T"] = s[:, 4].copy()
        return out

    def reset(self):
        for pr in self._probes:
            pr.reset()
        self._pending = 0
        self._t, self._series = [], []

    def close(self):
        for pr in self._probes:
            pr.close()



def particle_args(Ng, emitters, capacity, periodic, wall_mode, bins):
    """Checks of lbm.Particles' arguments -> (emitters float64 [E, 6], periodic_mask, bins uint32 [3]); ValueError for what luw_particles_create rejects."""
    Ng = np.asarray(Ng, np.int64)
    em = np.asarray(emitters, np.float64).reshape(-1, 6)
    per = [bool(v) for v in periodic]
    b = np.asarray(bins, np.int64).reshape(-1)
    if len(per) != 3 or b.size != 3:
        raise ValueError("periodic and bins take one value per axis")
    if int(capacity) < 1:
        raise ValueError("capacity must be at least 1")
    if int(wall_mode) not in (0, 1):
        raise ValueError("wall_mode must be 0 (reject the move) or 1 (deposit)")
    if (b < 1).any():
        raise ValueError("bin sizes must be at least 1")
    for a in range(3):
        if not per[a] and Ng[a] < 2:
            raise ValueError("a non-periodic axis needs at least 2 cells")
    if not np.isfinite(em).all() or (em[:, 3:] < 0).any():
        raise ValueError("emitter centres and half-extents must be finite, half-extents >= 0")
    for a in range(3):
        if not per[a] and ((em[:, a] - em[:, 3 + a] < 0) | (em[:, a] + em[:, 3 + a] > Ng[a] - 1)).any():
            raise ValueError("emitter boxes must lie inside [0, N-1] on non-periodic axes")
    return em, sum(1 << a for a in range(3) if per[a]), b.astype(np.uint32)


class Particles:
    """Lagrangian tracer particles in an in-process `LBM` of one domain (D == (1, 1, 1); a decomposed LBM raises ValueError, as particles crossing block
    faces would need a migration step). `emitters` [E, 6]: box centre x y z and half-extents x y z in global lattice coordinates; `capacity` ring slots;
    `periodic` one bool per axis (open faces elsewhere: a particle that leaves [0, N-1] becomes LEFT); wall_mode 0 rejects a move into a solid cell, 1 deposits
    the particle there; `seed` keys the random numbers; `bins` cells per concentration bin and axis. Everything is stream-ordered on the domain's stream;
    state() and bins() synchronise."""

    def __init__(self, lbm, emitters, capacity, periodic=(False, False, False), wall_mode=0, seed=0, bins=(1, 1, 1)):
        if tuple(lbm.D) != (1, 1, 1):
            raise ValueError("lbm.Particles needs a single domain, D == (1, 1, 1)")
        em, mask, b = particle_args(lbm.Ng, emitters, capacity, periodic, wall_mode, bins)
        self.lbm = lbm
        self._pt = DomainParticles(lbm.domains[0], em, int(capacity), mask, int(wall_mode), int(seed), b)

    def emit(self, per_emitter):
        self._pt.emit(per_emitter, t=self.lbm.t)

    def advance(self, dt=1.0, sigma=0.0):
        """One move with the lattice's current t, force and Coriolis."""
        lbm, d = self.lbm, self.lbm.domains[0]
        d.f, d.omega = lbm.f, lbm.omega
        self._pt.advance(dt, sigma, t=lbm.t)

    def count(self):
        self._pt.count()

    def state(self):
        return self._pt.state()

    def bins(self):
        return self._pt.bins()

    def reset_bins(self):
        self._pt.reset_bins()

    def close(self):
        self._pt.close()

class DistributedLBM(_Base):
    """One domain per rank (torch.distributed); rank r owns domain r of the split. Works with NCCL (GPU) and, for the host logic, with
    gloo: with `routing_only=True` no device domain is created and the class only does what is host logic -- the domain split, neighbour ranks, the
    x -> y -> z exchange order on host tensors -- while the caller supplies the extract / insert callbacks (the CPU tests plug the oracle in there).
    There is no CPU fallback of the LBM itself: initialize() / run() need the device domain."""

    def __init__(self, shape, D, group=None, device=0, routing_only=False, transport="ipc", **kw):
        super().__init__(shape, D, **kw)
        import torch
        import torch.distributed as dist
        self._torch, self._dist = torch, dist
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        assert self.world == len(self._split), "one rank per domain"
        self.d, self.O = self._split[self.rank]
        self.routing_only = bool(routing_only)
        self.device = device
        self.gidx = _local_index(self.Ng, self.Nl, self.O)
        if not self.routing_only:
            self.domain = self._make_domain(self.d, self.O, device)
            self.domains = [self.domain]
            # one explicit stream orders the step kernels, the halo kernels and the NCCL calls (torch's default stream has handle 0, which the C ABI
            # reads as "use the domain's own stream": kernels and NCCL would then run unordered on two streams)
            self._stream = torch.cuda.Stream(device=device)
            self.domain.set_stream(self._stream.cuda_stream)
            self.transport = transport
            if transport == "ipc":
                self._connect_ipc()
        else:
            self.domain, self.domains = None, []
        self._bufs = {}

    def _connect_ipc(self):
        """Exchange the CUDA IPC handles of the receive blocks (once) and map the two neighbours' blocks per decomposed axis. After this the
        step path makes no NCCL call: extract kernels store into the neighbours' memory over NVLink (luw_halo_ipc_exchange)."""
        dist = self._dist
        for axis in AXES:
            if self.D[axis] < 2:
                continue
            mine = self.domain.halo_ipc_export(axis)
            handles = [None] * self.world
            dist.all_gather_object(handles, mine, group=self.group)
            self.domain.halo_ipc_connect(axis, handles[self.rank_of(axis, +1)], handles[self.rank_of(axis, -1)])
        dist.barrier(group=self.group)

    def rank_of(self, axis, step):
        d = list(self.d)
        d[axis] = (d[axis] + step) % self.D[axis]
        return d[0] + self.D[0] * (d[1] + self.D[1] * d[2])

    def halo_bytes(self, payload, axis):
        A_ = (self.Nl[1] * self.Nl[2], self.Nl[2] * self.Nl[0], self.Nl[0] * self.Nl[1])[axis]
        ddf = 4 if self.precision == A.FP32 else 2
        per = {A.HALO_RHO_U_FLAGS: 17, A.HALO_FI: 5 * ddf, A.HALO_GI: ddf, A.HALO_T: 4}[payload]
        return per * A_

    def _buffers(self, payload, axis):
        key = (payload, axis)
        if key not in self._bufs:
            torch = self._torch
            dev = torch.device("cpu") if self.routing_only else torch.device("cuda", self.device)
            self._bufs[key] = tuple(torch.empty(self.halo_bytes(payload, axis), dtype=torch.uint8, device=dev) for _ in range(4))
        return self._bufs[key]

    def exchange(self, axis, sp, sm, rp, rm):
        """send_p -> (+) neighbour's recv_m, send_m -> (-) neighbour's recv_p. With 2 ranks on an axis both neighbours are the same rank."""
        dist = self._dist
        up, dn = self.rank_of(axis, +1), self.rank_of(axis, -1)
        if up == self.rank:  # a single domain on this axis never gets here; kept for completeness
            rm.copy_(sp); rp.copy_(sm)
            return
        ops = [dist.P2POp(dist.isend, sp, up, self.group, tag=2 * axis), dist.P2POp(dist.isend, sm, dn, self.group, tag=2 * axis + 1),
               dist.P2POp(dist.irecv, rm, dn, self.group, tag=2 * axis), dist.P2POp(dist.irecv, rp, up, self.group, tag=2 * axis + 1)]
        if not self.routing_only:
            with self._torch.cuda.stream(self._stream):  # NCCL enqueues on the current stream
                for r in dist.batch_isend_irecv(ops):
                    r.wait()
        else:
            for r in dist.batch_isend_irecv(ops):
                r.wait()

    def communicate(self, payload, extract, insert):
        for axis in AXES:
            if self.D[axis] < 2:
                continue
            if not self.routing_only and self.transport == "ipc":
                self.domain.halo_ipc_exchange(payload, axis)
                continue
            sp, sm, rp, rm = self._buffers(payload, axis)
            extract(payload, axis, sp, sm)
            self.exchange(axis, sp, sm, rp, rm)
            insert(payload, axis, rp, rm)

    # device-side callbacks
    def _extract(self, payload, axis, sp, sm):
        self.domain.halo_extract(payload, axis, sp.data_ptr(), sm.data_ptr())

    def _insert(self, payload, axis, rp, rm):
        self.domain.halo_insert(payload, axis, rp.data_ptr(), rm.data_ptr())

    def upload_slabs(self, slabs):
        """`slabs`: an iterable of (z0, flags, rho, u) pieces covering the local lattice plane range by plane range (z0 = first local z plane of the piece), uploaded
        as they come, so that a block of 10^9 cells never needs its 17 B per cell on the host. Follow with initialize() without images."""
        dom = self.domain
        plane, N = self.Nl[0] * self.Nl[1], dom.N
        for z0, fl, rh, uu in slabs:
            n = fl.size
            dom.upload_range(A.FIELD_FLAGS, fl, z0 * plane)
            dom.upload_range(A.FIELD_RHO, rh, z0 * plane)
            for c in range(3):
                dom.upload_range(A.FIELD_U, uu[c * n:(c + 1) * n], c * N + z0 * plane)
            dom.finish_queue()

    def initialize(self, flags=None, rho=None, u=None, T=None):
        """flags / rho / u (/ T with TEMPERATURE): LOCAL host images of this rank's domain (halo layers included); none at all after upload_slabs()."""
        if self.domain is None:
            raise RuntimeError("DistributedLBM(routing_only=True) has no device domain: the LBM step has no CPU fallback")
        dom = self.domain
        dom.f, dom.omega = self.f, self.omega
        if flags is None:
            pass  # the device fields are in place (upload_slabs)
        else:
            dom.rho[:], dom.u[:], dom.flags[:] = rho, u, flags
            if self.thermal and T is not None:
                dom.T[:] = T
            dom.upload_all()
        dom.t = 1
        self.communicate(A.HALO_RHO_U_FLAGS, self._extract, self._insert)
        dom.enqueue_initialize()
        self.communicate(A.HALO_RHO_U_FLAGS, self._extract, self._insert)
        self.communicate(A.HALO_FI, self._extract, self._insert)
        if self.thermal:
            self.communicate(A.HALO_T, self._extract, self._insert)
            self.communicate(A.HALO_GI, self._extract, self._insert)
        dom.finish_queue()
        dom.t = 0
        self.t = 0
        self.initialized = True

    def do_time_step(self):
        dom = self.domain
        if not self.routing_only and self.transport == "ipc":  # one call: step + exchanges, the y / z exchanges overlapped with the interior strips (luw_step_halo_ipc)
            dom.step_halo_ipc()
        else:
            dom.enqueue_stream_collide()
            self.communicate(A.HALO_FI, self._extract, self._insert)
            if self.thermal:
                self.communicate(A.HALO_GI, self._extract, self._insert)
        dom.increment_time_step()
        self.t += 1

    def run(self, steps=1):
        for _ in range(steps):
            self.do_time_step()

    def close(self):
        if self.domain is not None:
            self.domain.finish_queue()
            try:  # the neighbours store into this rank's IPC-mapped receive blocks: nobody frees before everybody has drained its stream
                self._dist.barrier(group=self.group)
            except Exception:
                pass
            self.domain.close()
            self.domain = None
