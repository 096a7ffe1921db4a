"""Host-side mirror of the reference's `LBM_Domain` (FX/lbm.hpp:26-221, FX/lbm.cpp:246-433) over the C ABI.

One Domain = one block of the lattice on one GPU: host mirrors of rho / u / flags (numpy, like Memory<T>'s host side,
FX/opencl.hpp:331-603), device buffers owned by the C library, and the enqueue_* calls of the reference under the same names.
"""
import ctypes as C

import numpy as np

from . import _cabi as A


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Domain:
    def __init__(self, Nx, Ny, Nz, D=(1, 1, 1), O=(0, 0, 0), precision=A.FP32, features=0, w=1.0, arith=A.ARITH_STRICT, device=0,
                 downstream_face=0, buffer_N=1, buffer_inv_tau=0.0, buffer_nudge_vertical=0, sponge_N=1, sponge_inv_tau=0.0):
        self.params = A.DomainParams(Nx, Ny, Nz, D[0], D[1], D[2], O[0], O[1], O[2], precision, features, arith, np.float32(w),
                                     downstream_face, buffer_N, np.float32(buffer_inv_tau), buffer_nudge_vertical, sponge_N,
                                     np.float32(sponge_inv_tau), device)
        self.Nx, self.Ny, self.Nz = Nx, Ny, Nz
        self.N = Nx * Ny * Nz
        self.precision = precision
        self.ddf_dtype = np.float32 if precision == A.FP32 else np.uint16
        self.t = 0
        self.f = (0.0, 0.0, 0.0)
        self.omega = (0.0, 0.0, 0.0)
        self._h = C.c_void_p()
        A.check(A.lib().luw_domain_create(C.byref(self.params), C.byref(self._h)))
        # host mirrors, initialised like the reference's Memory<> objects (rho=1, u=0, flags=0; FX/lbm.cpp:283-288) -- LAZILY: a mirror is allocated when the host
        # first touches it. The device fields hold the same values from luw_domain_create on, so an untouched mirror has nothing to upload; a case that moves its
        # boundary data through cell sets never owns a host image of the lattice (17 B per cell in the reference, FX/lbm.cpp:95-106).
        self._mirror = {}
        # thermal D3Q7 extension (features & TEMPERATURE): host mirror of T, 1 everywhere like Memory<float>(N, 1, .., 1.0f) (FX/lbm.cpp:323)
        self.thermal = bool(features & A.TEMPERATURE)

    _MIRRORS = {"rho": (A.FIELD_RHO, 1, np.float32, 1.0), "u": (A.FIELD_U, 3, np.float32, 0.0), "flags": (A.FIELD_FLAGS, 1, np.uint8, 0), "T": (A.FIELD_T, 1, np.float32, 1.0)}

    def _get_mirror(self, name):
        if name == "T" and not self.thermal:
            return None
        a = self._mirror.get(name)
        if a is None:
            _, comps, dtype, value = self._MIRRORS[name]
            a = np.full(comps * self.N, value, dtype) if value else np.zeros(comps * self.N, dtype)
            self._mirror[name] = a
        return a

    def _set_mirror(self, name, value):
        _, comps, dtype, _ = self._MIRRORS[name]
        if isinstance(value, np.ndarray) and value.dtype == dtype and value.size == comps * self.N and value.flags.c_contiguous:
            self._mirror[name] = value.reshape(-1)  # adopt the caller's buffer (e.g. page-locked memory) as the mirror
        else:
            self._get_mirror(name)[:] = value

    rho = property(lambda self: self._get_mirror("rho"), lambda self, v: self._set_mirror("rho", v))
    u = property(lambda self: self._get_mirror("u"), lambda self, v: self._set_mirror("u", v))
    flags = property(lambda self: self._get_mirror("flags"), lambda self, v: self._set_mirror("flags", v))
    T = property(lambda self: self._get_mirror("T"), lambda self, v: self._set_mirror("T", v))

    def host_mirror_bytes(self):
        """Bytes of host memory held by the mirrors that have been touched so far."""
        return sum(a.nbytes for a in self._mirror.values())

    def set_thermal(self, w_T, beta=0.0, T_avg=1.0):
        """def_w_T = 1/(2 alpha + 1/2), def_beta, def_T_avg (FX/lbm.cpp:750-752) for the launches that follow."""
        A.check(A.lib().luw_thermal_params(self._h, float(np.float32(w_T)), float(np.float32(beta)), float(np.float32(T_avg))))

    def read_gi(self):
        """Raw D3Q7 DDF image gi[i*N+n] (device-only in the reference; exposed for parity tests)."""
        out = np.empty(7 * self.N, self.ddf_dtype)
        A.check(A.lib().luw_download(self._h, A.FIELD_GI, _ptr(out), 0, out.size))
        self.finish_queue()
        return out

    # ---- lifetime
    def close(self):
        if self._h:
            A.lib().luw_domain_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- Memory<T>::enqueue_write_to_device / enqueue_read_from_device
    def _field(self, field):
        return {A.FIELD_RHO: self.rho, A.FIELD_U: self.u, A.FIELD_FLAGS: self.flags, A.FIELD_T: self.T}[field]

    def write_to_device(self, field, offset=0, count=None):
        host = self._field(field)
        count = host.size - offset if count is None else count
        A.check(A.lib().luw_upload(self._h, field, _ptr(host[offset:offset + count]), offset, count))

    def read_from_device(self, field, offset=0, count=None):
        host = self._field(field)
        count = host.size - offset if count is None else count
        A.check(A.lib().luw_download(self._h, field, _ptr(host[offset:offset + count]), offset, count))

    def upload_range(self, field, values, offset):
        """Elements [offset, offset + len(values)) of a field's dense host image, from a caller-owned array: lets a case that is generated slab by slab reach the
        device without a whole-field host image (luw_upload; pageable memory is staged before the call returns)."""
        values = np.ascontiguousarray(values)
        A.check(A.lib().luw_upload(self._h, field, _ptr(values), int(offset), int(values.size)))

    def _mirrored_fields(self):
        return (A.FIELD_RHO, A.FIELD_U, A.FIELD_FLAGS) + ((A.FIELD_T,) if self.thermal else ())

    def upload_all(self):
        names = {A.FIELD_RHO: "rho", A.FIELD_U: "u", A.FIELD_FLAGS: "flags", A.FIELD_T: "T"}
        for f in self._mirrored_fields():
            if names[f] in self._mirror:  # an untouched mirror equals what the device field was created with
                self.write_to_device(f)

    def download_all(self):
        for f in self._mirrored_fields():
            self.read_from_device(f)
        self.finish_queue()

    def read_fi(self):
        """Raw DDF image (device-only buffer in the reference; exposed for parity tests)."""
        out = np.empty(19 * self.N, self.ddf_dtype)
        A.check(A.lib().luw_download(self._h, A.FIELD_FI, _ptr(out), 0, out.size))
        self.finish_queue()
        return out

    def write_fi(self, fi):
        fi = np.ascontiguousarray(fi, self.ddf_dtype)
        assert fi.size == 19 * self.N
        A.check(A.lib().luw_upload(self._h, A.FIELD_FI, _ptr(fi), 0, fi.size))
        self.finish_queue()

    def device_ptr(self, field):
        p = C.c_void_p()
        A.check(A.lib().luw_device_ptr(self._h, field, C.byref(p)))
        return p.value

    # ---- kernels
    def enqueue_initialize(self):
        A.check(A.lib().luw_initialize(self._h))

    def enqueue_stream_collide(self):
        A.check(A.lib().luw_stream_collide(self._h, self.t, *map(float, self.f), *map(float, self.omega)))

    def enqueue_update_fields(self):
        A.check(A.lib().luw_update_fields(self._h, self.t, *map(float, self.f), *map(float, self.omega)))

    def run_steps(self, k):
        A.check(A.lib().luw_run_steps(self._h, self.t, k, *map(float, self.f), *map(float, self.omega)))
        self.t += k

    def increment_time_step(self, steps=1):
        self.t += steps

    def reset_time_step(self):
        self.t = 0

    def finish_queue(self):
        A.check(A.lib().luw_sync(self._h))

    def set_stream(self, cuda_stream):
        A.check(A.lib().luw_domain_set_stream(self._h, C.c_void_p(cuda_stream)))

    # ---- halo payloads (device buffers supplied by the caller as raw pointers)
    def halo_bytes(self, payload, axis):
        n = C.c_uint64()
        A.check(A.lib().luw_halo_bytes(self._h, payload, axis, C.byref(n)))
        return n.value

    def halo_extract(self, payload, axis, buf_p, buf_m):
        A.check(A.lib().luw_halo_extract(self._h, payload, axis, self.t, C.c_void_p(buf_p), C.c_void_p(buf_m)))

    def halo_insert(self, payload, axis, buf_p, buf_m):
        A.check(A.lib().luw_halo_insert(self._h, payload, axis, self.t, C.c_void_p(buf_p), C.c_void_p(buf_m)))

    def voxelize_mesh(self, direction, flag, p0, p1, p2, bbu):
        """LBM_Domain::voxelize_mesh_on_device -> run_voxelize_pass (FX/lbm.cpp:494-560) on the device flags / u; p0/p1/p2: 3 floats per triangle."""
        p0, p1, p2, bbu = (np.ascontiguousarray(a, np.float32) for a in (p0, p1, p2, bbu))
        A.check(A.lib().luw_voxelize_mesh(self._h, direction, flag, _ptr(p0), _ptr(p1), _ptr(p2), p0.size // 3, _ptr(bbu)))

    # ---- peer-mapped halo exchange of the one-process-per-GPU driver (CUDA IPC over NVLink)
    def halo_ipc_export(self, axis):
        h = C.create_string_buffer(64)
        A.check(A.lib().luw_halo_ipc_export(self._h, axis, h))
        return h.raw

    def halo_ipc_connect(self, axis, handle_up, handle_dn):
        A.check(A.lib().luw_halo_ipc_connect(self._h, axis, C.c_char_p(handle_up), C.c_char_p(handle_dn)))

    def halo_ipc_exchange(self, payload, axis):
        A.check(A.lib().luw_halo_ipc_exchange(self._h, payload, axis, self.t))

    def step_halo_ipc(self):
        """stream_collide + the fi (gi) exchanges of all decomposed axes, overlapped with the interior of the step where the decomposition allows it (luw_step_halo_ipc)."""
        A.check(A.lib().luw_step_halo_ipc(self._h, self.t, *map(float, self.f), *map(float, self.omega)))

    def overlapped_steps(self):
        n = C.c_uint64()
        A.check(A.lib().luw_overlapped_steps(self._h, C.byref(n)))
        return n.value

    # ---- measurement helpers
    def timer_begin(self):
        A.check(A.lib().luw_timer_begin(self._h))

    def timer_end(self):
        ms = C.c_float()
        A.check(A.lib().luw_timer_end(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self):
        n = C.c_uint64()
        A.check(A.lib().luw_launch_count(self._h, C.byref(n)))
        return n.value

    def uses_tiles(self):
        n = C.c_int()
        A.check(A.lib().luw_domain_step_kernel(self._h, C.byref(n)))
        return bool(n.value)

    def kernel_timing(self, enable):
        A.check(A.lib().luw_kernel_timing(self._h, int(bool(enable))))

    def kernel_timing_read(self):
        """(summed milliseconds, launches) of the main stream_collide kernel since the last read."""
        ms, n = C.c_float(), C.c_uint64()
        A.check(A.lib().luw_kernel_timing_read(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def column_ground(self):
        """-> uint32 [Ny, Nx]: global z of the lowest owned non-solid cell of every local column, 0xFFFFFFFF where there is none (luw_column_ground;
        read from the device flags, so no host mirror is touched)."""
        g = np.empty((self.Ny, self.Nx), np.uint32)
        A.check(A.lib().luw_column_ground(self._h, _ptr(g)))
        return g

    def solid_surface(self, periodic_mask=0):
        """-> uint64 local dense indices, ascending, of the owned solid cells with at least one counted link (luw_solid_surface; enumerated on the device).
        periodic_mask: bit a set = axis a is periodic (links across a global face of a non-periodic axis do not count)."""
        n = C.c_uint64()
        A.check(A.lib().luw_solid_surface(self._h, int(periodic_mask), 0, None, C.byref(n)))
        cells = np.empty(n.value, np.uint64)
        A.check(A.lib().luw_solid_surface(self._h, int(periodic_mask), cells.size, _ptr(cells), C.byref(n)))
        return cells

    def device_bytes(self):
        n = C.c_uint64()
        A.check(A.lib().luw_domain_bytes(self._h, C.byref(n)))
        return n.value


class VkInlet:
    """Device side of VonKarmanInletUpdater (FX/setup.cpp:1034-1086, kernel FX/kernel.cpp:2495-2571)."""

    def __init__(self, domain, point_cell, point_face, point_data, mode_data, mode_count, mode_stride):
        self.domain = domain
        self._h = C.c_void_p()
        pc = np.ascontiguousarray(point_cell, np.uint64)
        pf = np.ascontiguousarray(point_face, np.uint8)
        pd = np.ascontiguousarray(point_data, np.float32)
        md = np.ascontiguousarray(mode_data, np.float32)
        assert pd.size == 7 * pc.size and md.size == 10 * mode_stride
        A.check(A.lib().luw_vk_inlet_create(domain._h, pc.size, mode_count, mode_stride, _ptr(pc), _ptr(pf), _ptr(pd), _ptr(md), C.byref(self._h)))

    def apply(self, use_interp, t0, t1, alpha):
        A.check(A.lib().luw_vk_inlet_apply(self._h, int(use_interp), float(t0), float(t1), float(alpha)))

    def close(self):
        if self._h:
            A.lib().luw_vk_inlet_destroy(self._h)
            self._h = C.c_void_p()


class CellSet:
    """A fixed list of local cells whose rho / u / flags are uploaded or read back without moving the whole field (boundary-field upload,
    probes). Values are SoA over the set: [c*count + k]."""

    def __init__(self, domain, cells):
        self.domain = domain
        self.cells = np.ascontiguousarray(cells, np.uint64)
        self.count = int(self.cells.size)
        self._h = C.c_void_p()
        A.check(A.lib().luw_cellset_create(domain._h, self.count, _ptr(self.cells), C.byref(self._h)))

    def upload(self, field, values):
        A.check(A.lib().luw_cellset_upload(self._h, field, _ptr(values)))

    def download(self, field, values):
        A.check(A.lib().luw_cellset_download(self._h, field, _ptr(values)))

    def close(self):
        if self._h:
            A.lib().luw_cellset_destroy(self._h)
            self._h = C.c_void_p()


class Stats:
    """Device-side running mean / M2 of u and mean of rho (luw_stats_*): the reference's accumulate_from_buffers (FX/setup.cpp:4441-4488) without the
    per-sample full-field read-back."""

    def __init__(self, domain):
        self.domain = domain
        self._h = C.c_void_p()
        A.check(A.lib().luw_stats_create(domain._h, C.byref(self._h)))

    def accumulate(self):
        A.check(A.lib().luw_stats_accumulate(self._h))

    def reset(self):
        A.check(A.lib().luw_stats_reset(self._h))

    def download(self):
        """-> (mean_u[3N] SoA, m2_u[3N] SoA, mean_rho[N], count)"""
        N = self.domain.N
        mean_u, m2_u, mean_rho = np.empty(3 * N, np.float32), np.empty(3 * N, np.float32), np.empty(N, np.float32)
        n = C.c_uint64()
        A.check(A.lib().luw_stats_download(self._h, _ptr(mean_u), _ptr(m2_u), _ptr(mean_rho), C.byref(n)))
        return mean_u, m2_u, mean_rho, n.value

    def download_T(self):
        """-> mean_T[N] (LUW_TEMPERATURE domains: the reference's avg_T, FX/setup.cpp:4481-4486)"""
        mean_T = np.empty(self.domain.N, np.float32)
        A.check(A.lib().luw_stats_download_temperature(self._h, _ptr(mean_T)))
        return mean_T

    def close(self):
        if self._h:
            A.lib().luw_stats_destroy(self._h)
            self._h = C.c_void_p()


class WindStats:
    """Pedestrian-level wind statistics of a fixed list of local cells (luw_wind_stats_*): running means and co-moments of u, mean / M2 / peak of the speed
    and threshold exceedance counts, accumulated on the device once per sample. `thresholds`: speeds in lattice units (at most 8)."""

    def __init__(self, domain, cells, thresholds=()):
        self.domain = domain
        self.cells = np.ascontiguousarray(cells, np.uint64)
        self.count = int(self.cells.size)
        self.thresholds = np.ascontiguousarray(thresholds, np.float32)
        self._h = C.c_void_p()
        A.check(A.lib().luw_wind_stats_create(domain._h, self.count, _ptr(self.cells), int(self.thresholds.size), _ptr(self.thresholds), C.byref(self._h)))

    def accumulate(self):
        A.check(A.lib().luw_wind_stats_accumulate(self._h))

    def reset(self):
        A.check(A.lib().luw_wind_stats_reset(self._h))

    def download(self):
        """-> (mean_u[3, count], comoment[6, count] (uu vv ww uv uw vw), mean_speed[count], m2_speed[count], max_speed[count], exceed[thresholds, count], samples)"""
        K, T = self.count, int(self.thresholds.size)
        mean_u, com = np.empty((3, K), np.float32), np.empty((6, K), np.float32)
        ms, m2, mx = np.empty(K, np.float32), np.empty(K, np.float32), np.empty(K, np.float32)
        ex = np.empty((T, K), np.uint32)
        n = C.c_uint64()
        A.check(A.lib().luw_wind_stats_download(self._h, _ptr(mean_u), _ptr(com), _ptr(ms), _ptr(m2), _ptr(mx), _ptr(ex), C.byref(n)))
        return mean_u, com, ms, m2, mx, ex, n.value

    def close(self):
        if self._h:
            A.lib().luw_wind_stats_destroy(self._h)
            self._h = C.c_void_p()


class WallLoads:
    """Wind loads of a list of local solid cells (luw_wall_loads_*): per sample and label the sums of the momentum-exchange force F and of its moment
    (r - r0) x F in double, kept in a device ring of `capacity` samples until drained, and per cell the running mean / M2 of F. `cells` / `labels` sorted by
    (label, index); ref_points [L, 3] (global lattice coordinates)."""

    def __init__(self, domain, cells, labels, label_count, ref_points, periodic_mask=0, capacity=256):
        self.domain = domain
        self.cells = np.ascontiguousarray(cells, np.uint64)
        self.labels = np.ascontiguousarray(labels, np.uint32)
        self.count, self.L, self.capacity = int(self.cells.size), int(label_count), int(capacity)
        self.ref_points = np.ascontiguousarray(ref_points, np.float64)
        assert self.labels.size == self.count and self.ref_points.size == 3 * self.L
        self._h = C.c_void_p()
        A.check(A.lib().luw_wall_loads_create(domain._h, self.count, _ptr(self.cells), _ptr(self.labels), self.L, _ptr(self.ref_points), int(periodic_mask),
                                              self.capacity, C.byref(self._h)))

    def accumulate(self, t=None):
        """One sample of the current state (t: the domain's time step by default). Stream-ordered, no synchronisation."""
        A.check(A.lib().luw_wall_loads_accumulate(self._h, self.domain.t if t is None else int(t)))

    def drain(self):
        """-> float64 [samples, L, 6] (Fx Fy Fz Mx My Mz) of the pending samples, in order; synchronous; clears them."""
        out = np.empty((self.capacity, self.L, 6), np.float64)
        n = C.c_uint64()
        A.check(A.lib().luw_wall_loads_drain(self._h, _ptr(out), C.byref(n)))
        return out[:n.value].copy()

    def download_cells(self):
        """-> (mean_F [3, count], m2_F [3, count], samples since create / reset)"""
        mean, m2 = np.empty((3, self.count), np.float32), np.empty((3, self.count), np.float32)
        n = C.c_uint64()
        A.check(A.lib().luw_wall_loads_download_cells(self._h, _ptr(mean), _ptr(m2), C.byref(n)))
        return mean, m2, n.value

    def reset(self):
        A.check(A.lib().luw_wall_loads_reset(self._h))

    def close(self):
        if self._h:
            A.lib().luw_wall_loads_destroy(self._h)
            self._h = C.c_void_p()


def pinned_empty(count, dtype):
    """numpy array over page-locked host memory (luw_host_alloc). The array keeps the allocation alive through its base object."""
    dtype = np.dtype(dtype)
    nbytes = int(count) * dtype.itemsize
    p = C.c_void_p()
    A.check(A.lib().luw_host_alloc(C.byref(p), max(nbytes, 1)))

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                A.lib().luw_host_free(self.ptr)
            except Exception:
                pass

    buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
    buf._owner = _Owner(p)  # the ctypes array accepts attributes; numpy keeps `buf` alive as the base of the returned array
    return np.frombuffer(buf, dtype=dtype, count=int(count))
