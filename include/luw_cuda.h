/* luw_cuda.h -- C ABI of the B200 (sm_100a) implementation of LatticeUrbanWind's LBM time step.
 *
 * This is the drop-in seam. In the reference the LBM host layer (FX/lbm.cpp, class LBM_Domain) reaches the device only through
 * Device / Memory<T> / Kernel of FX/opencl.hpp:274-683 and the OpenCL-C program of FX/kernel.cpp. Every entry point below replaces
 * one of those interactions; the citation next to it names the reference call it stands in for
 * (FX = core/cfd_core/FluidX3D/src of hweifluids/LatticeUrbanWind).
 *
 * Conventions
 *  - plain C types only; all pointers named `host_*` are host memory, `dev_*` are device memory of the domain's GPU;
 *  - every function returns 0 on success, otherwise a luw_status code; luw_last_error_string() describes the last failure of the
 *    calling thread. The reference prints and exit(1)s on any device error (FX/utilities.hpp:4370-4382, FX/opencl.hpp:613-618);
 *    the C++ host layer (latticeurbanwind_b200/host/lbm.hpp) converts a non-zero status into the same print_error + exit(1);
 *  - all work of a domain is enqueued on that domain's stream (luw_domain_set_stream) and is asynchronous unless stated;
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with LUW_ERR_NO_DEVICE.
 *
 * Memory layout of every HOST image and of every element range / cell index that crosses this interface (identical to the reference,
 * FX/kernel.cpp:833-839,877-879): SoA, n = x + (y + z*Ny)*Nx over the LOCAL lattice including halo layers; fi[i*N + n] (i = 0..18, float /
 * IEEE half scaled by 2^15 / custom 1-4-11 half), u[c*N + n], rho[n], flags[n]. On the device the rows are padded to a multiple of 16
 * elements (row pitch Px >= Nx, component stride Px*Ny*Nz) so that TMA can address any lattice, e.g. the Nx/Dx + 2 cells of an x-decomposed
 * block; luw_upload / luw_download / cell sets / inlet points translate. Only luw_device_ptr exposes the pitched arrays.
 */
#ifndef LUW_CUDA_H
#define LUW_CUDA_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum luw_status {
	LUW_OK = 0,
	LUW_ERR_INVALID = 1, /* bad argument / unsupported combination */
	LUW_ERR_NO_DEVICE = 2, /* no CUDA device or driver */
	LUW_ERR_OOM = 3, /* cudaMalloc failed (reference: predicted before allocation, FX/opencl.hpp:364-365) */
	LUW_ERR_CUDA = 4 /* any other CUDA runtime error */
} luw_status;

/* DDF storage precision: compile-time FP16S / FP16C / (none) in FX/defines.hpp:13-14, `fpxx` in FX/defines.hpp:68-72 */
enum { LUW_FP32 = 0, LUW_FP16S = 1, LUW_FP16C = 2 };
/* extension switches: compile-time in the reference (FX/defines.hpp:17-29; BUFFER_NUDGING / TOP_SPONGE FX/lbm.cpp:770-782) */
enum {
	LUW_UPDATE_FIELDS = 1u, LUW_VOLUME_FORCE = 2u, LUW_EQUILIBRIUM_BOUNDARIES = 4u, LUW_SUBGRID = 8u,
	LUW_BUFFER_NUDGING = 16u, LUW_TOP_SPONGE = 32u,
	LUW_TEMPERATURE = 64u /* thermal D3Q7 transport (FX/defines.hpp:23): allocates gi (7 fpxx per cell) and T (1 float per cell), see luw_thermal_params */
};
/* arithmetic policy of the step kernels */
enum {
	LUW_ARITH_STRICT = 0, /* "as written": fused only where the reference writes fma(), IEEE div/sqrt -> bit-identical to oracle/ */
	LUW_ARITH_FAST = 1 /* mul+add contraction and approximate reciprocals allowed (what -cl-mad-enable licenses, FX/opencl.hpp:305) */
};
enum { LUW_FIELD_RHO = 0, LUW_FIELD_U = 1, LUW_FIELD_FLAGS = 2, LUW_FIELD_FI = 3, LUW_FIELD_T = 4, LUW_FIELD_GI = 5 /* T[n], gi[i*N+n] i = 0..6: LUW_TEMPERATURE domains */ };
/* halo payloads: enum_transfer_field of FX/lbm.hpp:24 (fi: 5 DDFs per face cell; rho_u_flags: 17 bytes per face cell; gi: 1 DDF per face cell; T: 1 float) */
enum { LUW_HALO_FI = 0, LUW_HALO_RHO_U_FLAGS = 1, LUW_HALO_GI = 2, LUW_HALO_T = 3 };

typedef struct luw_device_info { /* subset of Device_Info, FX/opencl.hpp:89-188, used by device selection and the info printout */
	char name[256];
	uint64_t memory_bytes;
	uint32_t compute_units; /* SMs */
	uint32_t clock_mhz;
	uint32_t cc_major, cc_minor;
} luw_device_info;

typedef struct luw_domain_params { /* LBM_Domain ctor arguments (FX/lbm.cpp:235-281) + the def_* constants of FX/lbm.cpp:612-783 */
	uint32_t Nx, Ny, Nz; /* local lattice incl. halo layers */
	uint32_t Dx, Dy, Dz; /* domains per axis (halo layers exist on axes with D>1) */
	int32_t Ox, Oy, Oz; /* global coordinate of local cell 0 */
	uint32_t precision; /* LUW_FP32 / LUW_FP16S / LUW_FP16C */
	uint32_t features; /* LUW_* extension bits */
	uint32_t arith; /* LUW_ARITH_STRICT / LUW_ARITH_FAST */
	float w; /* def_w = 1/tau as the kernel sees it */
	int32_t downstream_face; /* def_downstream_face: 0 none, 1 west, 2 east, 3 south, 4 north */
	uint32_t buffer_N; float buffer_inv_tau; int32_t buffer_nudge_vertical; /* BUFFER_NUDGING constants */
	uint32_t sponge_N; float sponge_inv_tau; /* TOP_SPONGE constants (sponge_ref_mode 0) */
	int32_t device; /* CUDA device ordinal */
} luw_domain_params;

typedef struct luw_domain luw_domain; /* opaque: stands for one LBM_Domain's device side (Device + Memory<> + Kernel objects) */
typedef struct luw_vk_inlet luw_vk_inlet; /* opaque: device buffers + kernel of VonKarmanInletUpdater (FX/setup.cpp:1034-1086) */

const char* luw_last_error_string(void);

/* get_devices() / Device_Info, FX/opencl.hpp:212-242 */
int luw_device_count(int* count);
int luw_get_device_info(int device, luw_device_info* info);

/* LBM_Domain::LBM_Domain + allocate(): FX/lbm.cpp:235-338 (Memory<> ctors allocate and zero-fill, FX/opencl.hpp:383-391) */
int luw_domain_create(const luw_domain_params* params, luw_domain** out);
int luw_domain_destroy(luw_domain* dom); /* ~LBM_Domain / Memory<> dtors */
/* use an existing CUDA stream (cudaStream_t passed as void*) for everything the domain enqueues; NULL restores the domain's own stream */
int luw_domain_set_stream(luw_domain* dom, void* cuda_stream);
int luw_domain_bytes(const luw_domain* dom, uint64_t* device_bytes); /* Device_Info::memory_used, FX/info.cpp:233-241 */
/* which stream_collide implementation the domain runs: 1 = TMA-tiled persistent kernel (lattices with an even x extent of at least one 64-cell
 * tile), 0 = one-cell-per-thread kernel (any lattice). Same results; the reference has a single kernel (FX/kernel.cpp:1475). */
int luw_domain_step_kernel(const luw_domain* dom, int* tiled);

/* Memory<T>::enqueue_write_to_device / enqueue_read_from_device(offset,length): FX/opencl.hpp:481-512. offset/count in ELEMENTS of the field
 * (rho: N floats, u: 3N floats, flags: N bytes, fi: 19N fpxx). Host pointers may be pageable or pinned; copies are stream-ordered. */
int luw_upload(luw_domain* dom, int field, const void* host_src, uint64_t offset, uint64_t count);
int luw_download(luw_domain* dom, int field, void* host_dst, uint64_t offset, uint64_t count);
int luw_device_ptr(luw_domain* dom, int field, void** dev_ptr); /* raw device pointer of a field (pitched rows, see above) */

/* Thermal D3Q7 extension (SURVEY.md 8-f4). A domain created with LUW_TEMPERATURE runs the reference's TEMPERATURE blocks inside initialize /
 * stream_collide / update_fields (FX/kernel.cpp:1306-1336, 1442-1450, 1639-1684, 1981-2000): cells flagged TYPE_T (0x04) hold their preset T, every other
 * fluid cell transports T with a D3Q7 SRT collision at rate w_T, relaxes it towards the top row inside the TOP_SPONGE zone, and (VOLUME_FORCE) feels the
 * buoyancy -f*beta*(T-T_avg). Constants: def_w_T = 1/(2 alpha + 1/2), def_beta, def_T_avg of FX/lbm.cpp:750-752 (LBM ctor arguments alpha, beta;
 * T_avg = 1). Defaults w_T = 1, beta = 0, T_avg = 1. T starts at 1 like Memory<float>(N, 1, .., 1.0f) (FX/lbm.cpp:323); upload it before luw_initialize.
 * Decomposed runs exchange LUW_HALO_GI after LUW_HALO_FI every step and LUW_HALO_T + LUW_HALO_GI at the end of initialisation (FX/lbm.cpp LBM::initialize /
 * do_time_step); luw_run_steps_multi does the per-step part. These domains use the one-cell-per-thread step kernel (luw_domain_step_kernel reports 0). */
int luw_thermal_params(luw_domain* dom, float w_T, float beta, float T_avg);

/* kernel "initialize", FX/kernel.cpp:1370-1452, enqueued by LBM_Domain::enqueue_initialize FX/lbm.cpp:340-343 (slot parity t=1 baked in) */
int luw_initialize(luw_domain* dom);
/* kernel "stream_collide", FX/kernel.cpp:1475-1780, enqueued by LBM_Domain::enqueue_stream_collide FX/lbm.cpp:344-346 with (t,fx,fy,fz,omega) */
int luw_stream_collide(luw_domain* dom, uint64_t t, float fx, float fy, float fz, float omega_x, float omega_y, float omega_z);
/* kernel "update_fields", FX/kernel.cpp:1938-2028, enqueued by LBM_Domain::enqueue_update_fields FX/lbm.cpp:348-355 */
int luw_update_fields(luw_domain* dom, uint64_t t, float fx, float fy, float fz, float omega_x, float omega_y, float omega_z);
/* k consecutive single-domain steps t0..t0+k-1 without host round trips: the body of LBM::run for D==1 (FX/lbm.cpp:1262-1312) minus its per-step finish() */
int luw_run_steps(luw_domain* dom, uint64_t t0, uint64_t k, float fx, float fy, float fz, float omega_x, float omega_y, float omega_z);

/* kernels "transfer_extract_*" / "transfer__insert_*", FX/kernel.cpp:2241-2310, enqueued by enqueue_transfer_extract/insert_field FX/lbm.cpp:1895-1906.
 * axis 0/1/2 = x/y/z. dev_buf_p / dev_buf_m are DEVICE buffers of luw_halo_bytes() bytes each, laid out [b*A + a] like the reference's transfer buffers;
 * who moves them between domains (peer copy, NCCL) is the caller's business -- that replaces the host-staged swap of FX/lbm.cpp:1907-1935. */
int luw_halo_bytes(const luw_domain* dom, int payload, uint32_t axis, uint64_t* bytes);
int luw_halo_extract(luw_domain* dom, int payload, uint32_t axis, uint64_t t, void* dev_buf_p, void* dev_buf_m);
int luw_halo_insert(luw_domain* dom, int payload, uint32_t axis, uint64_t t, const void* dev_buf_p, const void* dev_buf_m);

/* LBM::communicate_field, FX/lbm.cpp:1907-1935, for ALL domains of a decomposition that live in this process: `doms[d]`, d = dx + (dy + dz*Dy)*Dx,
 * count = Dx*Dy*Dz. For the given axis: extract on every domain, device-to-device (peer) copies of the two face payloads to the periodic neighbours
 * (d +- 1) % D, insert on every domain -- all asynchronous on the domains' streams, ordered by events; no host staging, no host synchronisation.
 * Axes must be exchanged in the order x, y, z (edge / corner DDFs travel through two hops, like in the reference). */
int luw_halo_exchange(luw_domain* const* doms, uint32_t count, int payload, uint32_t axis, uint64_t t);
/* LBM::communicate_field, FX/lbm.cpp:1907-1935, for the one-process-per-GPU driver (every rank owns ONE domain of the decomposition; all ranks on one
 * NVLink / NVSwitch node). The receive buffers of a domain are exported with CUDA IPC; a neighbour maps them and its extract kernel stores the face payload
 * straight into them over NVLink (no staging copy, no NCCL call on the step path), then raises a sequence flag in the same mapping; the receiver's stream
 * waits for the flags of both neighbours and runs the insert kernel. Two buffer sets alternate, which is enough because a rank cannot start exchange s+2
 * on an axis before its neighbours have finished inserting exchange s (their exchange s+1, which this rank waits for, is enqueued after it).
 *   export:   allocates the axis' receive block and writes its 64-byte cudaIpcMemHandle_t to `handle_out`;
 *   connect:  maps the blocks of the (+) and the (-) neighbour rank (the two handles are equal when the axis has two domains);
 *   exchange: extract -> remote stores -> signal -> wait -> insert, all enqueued on the domain's stream; every rank must issue the same sequence of
 *             exchanges per axis (payloads may alternate: rho_u_flags at initialisation, fi every step). Axes in the order x, y, z. */
int luw_halo_ipc_export(luw_domain* dom, uint32_t axis, void* handle_out);
int luw_halo_ipc_connect(luw_domain* dom, uint32_t axis, const void* handle_up, const void* handle_dn);
int luw_halo_ipc_exchange(luw_domain* dom, int payload, uint32_t axis, uint64_t t);
/* One time step of a rank of the one-process-per-GPU driver: stream_collide + the fi (and gi) exchanges of every decomposed axis, x -> y -> z (do_time_step +
 * communicate_fi, FX/lbm.cpp:1262-1290, 1907-1935) -- with the exchange OVERLAPPED with the interior of the step where the decomposition allows it (y / z splits of a
 * TMA-tiled domain): the step kernel collides the strips that hold the halo / boundary layers first and counts them as they reach global memory; a second stream waits
 * for that count and runs extract -> remote store -> flag -> wait -> insert while the interior strips are still being collided; the domain's stream waits for the
 * insert before anything else. Same results, bit for bit, as luw_stream_collide followed by luw_halo_ipc_exchange per axis (which is what it does when x is
 * decomposed -- x faces involve every strip --, for thermal domains, or with LUW_HALO_OVERLAP=0). */
int luw_step_halo_ipc(luw_domain* dom, uint64_t t, float fx, float fy, float fz, float omega_x, float omega_y, float omega_z);
int luw_overlapped_steps(const luw_domain* dom, uint64_t* steps); /* how many luw_step_halo_ipc calls ran their exchange overlapped with the step (diagnostics, tests) */
/* LBM::do_time_step for `k` steps t0..t0+k-1 on all domains of a decomposition (FX/lbm.cpp:1262-1290): stream_collide on every domain, then
 * luw_halo_exchange(HALO_FI) for x, y, z. The reference's per-step finish_queue / barriers are gone: everything is stream-ordered. */
int luw_run_steps_multi(luw_domain* const* doms, uint32_t count, uint64_t t0, uint64_t k, float fx, float fy, float fz, float omega_x, float omega_y, float omega_z);

/* kernel "vk_inlet_apply", FX/kernel.cpp:2495-2571; buffers as packed by VonKarmanInletUpdater (FX/setup.cpp:886-1116):
 * point_cell[P] u64 local cell index, point_face[P] u8, point_data[7*P] f32 SoA (px,py,pz,ubx,uby,ubz,sigma), mode_data[10*V] f32 SoA */
int luw_vk_inlet_create(luw_domain* dom, uint64_t point_count, uint64_t mode_count, uint64_t mode_stride,
	const uint64_t* host_point_cell, const uint8_t* host_point_face, const float* host_point_data, const float* host_mode_data, luw_vk_inlet** out);
int luw_vk_inlet_apply(luw_vk_inlet* vk, uint32_t use_interp, float t0, float t1, float alpha);
int luw_vk_inlet_destroy(luw_vk_inlet* vk);

/* kernel "voxelize_mesh", FX/kernel.cpp:2381-2471, as launched by LBM_Domain::voxelize_mesh_on_device -> run_voxelize_pass (FX/lbm.cpp:494-560): rays along
 * `direction` (0/1/2 = x/y/z; LUW voxelises TYPE_S geometry along z, FX/lbm.cpp:585-587) through every column of the domain, flags of the cells inside the
 * closed triangle mesh get `flag`, previously solid cells outside are released. host_p0/p1/p2: 3 floats per triangle in lattice coordinates (the mesh as
 * FX/setup.cpp:4084-4087 leaves it); host_bbu: the 16 floats of `bounding_box_and_velocity` (FX/lbm.cpp:529-549: triangle count as float bits, bounding
 * box -+ 2 cells, rotation centre, linear and rotational velocity). Only resting geometry (velocities 0, the only way LUW calls it) is supported:
 * otherwise LUW_ERR_INVALID. Works on the device flags / u in place (upload the host images first if they were edited); bit-exact with the reference. */
int luw_voxelize_mesh(luw_domain* dom, uint32_t direction, uint8_t flag, const float* host_p0, const float* host_p1, const float* host_p2, uint32_t triangle_count, const float* host_bbu);

/* Boundary-field evaluation (SURVEY.md 8-f2): the sample searches of the reference's inflow interpolators, one open-face cell per GPU thread; bit-exact with the
 * host code (same sequential algorithm per cell, individually rounded float operations). Host buffers in and out; synchronous. The cells are the TYPE_E cells of the five
 * open faces the reference finds by visiting every lattice cell (apply_inlet_outlet, FX/interpolation.cpp:66-210; apply_inlet_outlet_hd, FX/interpolation_hd.cpp:443-750).
 * luw_inlet_nearest: NearestNeighborInterpolator::eval (FX/interpolation.cpp:53-62). host_cell_xyz: x[n] y[n] z[n] (SoA); host_point_xyz: x, y, z per sample;
 *   host_nearest[c] = index of the first sample at the smallest squared distance, 0xFFFFFFFF if there is none (the reference then leaves u = 0).
 * luw_inlet_knn: the K = 64 selection loop of KNNInterpolatorHD::eval (FX/interpolation_hd.cpp:232-296) for cells that lie on one face plane. host_point_ab: the
 *   in-plane coordinates (a, b) of the samples on that plane, in sample order; host_cell_ab: a[n] b[n]. Per cell: host_exact[c] = first sample within 1e-16 (squared)
 *   of the cell, else -1; host_used[c] <= 64 samples kept, host_kept[64*c + k] their indices in the reference's slot order (the order of its double-precision sums),
 *   host_max_r2[c] = max_r2_kept. The weighted quadratic fit over the kept samples (FX/interpolation_hd.cpp:298-410) is the caller's, on the host: its weights are
 *   exp() in double and must come from the host's libm to reproduce the reference's bits (latticeurbanwind_b200/host/inlet_outlet_surface.cpp). */
#define LUW_INLET_KNN_K 64
int luw_inlet_nearest(int device, uint64_t cell_count, const float* host_cell_xyz, uint32_t point_count, const float* host_point_xyz, uint32_t* host_nearest);
int luw_inlet_knn(int device, uint64_t cell_count, const float* host_cell_ab, uint32_t point_count, const float* host_point_ab,
	uint32_t* host_kept, uint32_t* host_used, float* host_max_r2, int32_t* host_exact);
int luw_inlet_launch_count(uint64_t* launches); /* kernels launched by the two calls above in this process (diagnostics, tests) */

/* Boundary-field upload and probe read-back without moving whole fields. The reference writes boundary values into the full host mirrors and
 * uploads / downloads ALL N cells (LBM::initialize FX/lbm.cpp:1226-1237; probes and sampling read the whole u field back, FX/setup.cpp:4411-4425,
 * 4498-4509). A cell set is a fixed list of local cell indices (e.g. the TYPE_E inflow faces, a probe plane); upload scatters host values
 * [c*count + k] (c = component: rho 1, u 3, flags 1) into the field, download gathers them. Host buffers may be pinned (luw_host_alloc). */
typedef struct luw_cellset luw_cellset;
int luw_cellset_create(luw_domain* dom, uint64_t count, const uint64_t* host_cell_index, luw_cellset** out);
int luw_cellset_upload(luw_cellset* set, int field, const void* host_values);
int luw_cellset_download(luw_cellset* set, int field, void* host_values);
int luw_cellset_destroy(luw_cellset* set);

/* Device-side time averaging (SURVEY.md 8-f3). The reference reads u and rho of ALL cells back every sample and updates running mean / M2 on host threads
 * (process_post_step_samples -> enqueue_read_u_rho + accumulate_from_buffers, FX/setup.cpp:4411-4425, 4441-4488, 4510-4542). Here the accumulators live in
 * HBM and one kernel applies the same per-cell Welford update (same operations, same roundings) to the fields where they are; only the finished
 * statistics cross PCIe. accumulate: ++count, inv_n = 1/count, mean += (x-mean)*inv_n, M2 += (x-mean_old)*(x-mean_new) for ux, uy, uz; running mean of rho.
 * The caller runs luw_update_fields first when the domain does not store rho/u every step, like the reference does (FX/setup.cpp:4412-4414).
 * download: dense host arrays in the layout of `u` / `rho`: mean_u[c*N+n], m2_u[c*N+n] (c = 0..2), mean_rho[n]; any pointer may be NULL.
 * (The reference keeps avg_u interleaved [3n+c] and M2 per component; the C++ host layer re-packs, latticeurbanwind_b200/host/lbm.hpp.) */
typedef struct luw_stats luw_stats;
int luw_stats_create(luw_domain* dom, luw_stats** out); /* accumulators zero-filled: avg_u.assign(.., 0.0f) ..., FX/setup.cpp:4258-4266 */
int luw_stats_accumulate(luw_stats* st);
int luw_stats_reset(luw_stats* st); /* std::fill(.., 0.0f), avg_count = 0: FX/setup.cpp:4556-4562 */
int luw_stats_download(luw_stats* st, float* host_mean_u, float* host_m2_u, float* host_mean_rho, uint64_t* count);
/* LUW_TEMPERATURE domains: accumulate also keeps the running mean of T (avg_T under `include_temperature_avg`, FX/setup.cpp:4449-4451, 4481-4486); dense host array [n] */
int luw_stats_download_temperature(luw_stats* st, float* host_mean_T);
int luw_stats_destroy(luw_stats* st);

/* Pedestrian-level wind statistics. Extends the averaging window above (FX/setup.cpp:4411-4542) and what write_avg_vtk derives from it (TKE / TI from mean and
 * M2 per component, FX/setup.cpp:2513-2683) with quantities that cannot be rebuilt from those accumulators; the reference has NO counterpart (it would read the whole
 * u field back per sample and loop on the host). The accumulators cover a fixed list of cells only -- typically a few layers at fixed heights above the local
 * ground or roof -- so they stay small on any lattice.
 * luw_column_ground: host_ground[y*Nx + x] over the local Nx*Ny columns = GLOBAL z (Oz + z) of the lowest owned cell (z halo layers skipped) whose flags are not
 *   solid ((flags & 0x03) != TYPE_S), 0xFFFFFFFF if the column has none; read from the device flags; synchronous. Over a decomposition in z the ground of a global
 *   column is the minimum over its blocks.
 * luw_wind_stats_create: host_cell_index[count] = local dense cell indices (like luw_cellset_create); host_thresholds: speeds in lattice units (>= 0, at most
 *   LUW_WIND_MAX_THRESHOLDS). Accumulators zero-filled; count may be 0.
 * luw_wind_stats_accumulate: ++n, inv_n = 1/n; per listed cell the Welford update of the means of ux, uy, uz and of their co-moments
 *   C_ab += (x_a - mean_a,old)*(x_b - mean_b,new), ab = uu vv ww uv uw vw (C_ab / n is the covariance, u'w' = C_uw / n), Welford mean / M2 of the speed
 *   s = |u|, its running maximum (from 0) and, per threshold, the number of samples with s > threshold. Every product and sum is rounded separately, so the
 *   means and C_uu / C_vv / C_ww equal luw_stats' mean_u / m2_u for the same cells bit for bit. Stream-ordered on the domain's stream, no host synchronisation;
 *   the caller runs luw_update_fields first when the domain does not store u every step, like for luw_stats_accumulate.
 * luw_wind_stats_download: SoA over the list [j*count + k]: mean_u 3*count (u v w), comoment 6*count (uu vv ww uv uw vw), mean_speed / m2_speed / max_speed count
 *   each, exceed threshold_count*count; any pointer may be NULL; synchronous. */
#define LUW_WIND_MAX_THRESHOLDS 8
typedef struct luw_wind_stats luw_wind_stats;
int luw_column_ground(luw_domain* dom, uint32_t* host_ground);
int luw_wind_stats_create(luw_domain* dom, uint64_t count, const uint64_t* host_cell_index, uint32_t threshold_count, const float* host_thresholds, luw_wind_stats** out);
int luw_wind_stats_accumulate(luw_wind_stats* st);
int luw_wind_stats_reset(luw_wind_stats* st);
int luw_wind_stats_download(luw_wind_stats* st, float* host_mean_u, float* host_comoment, float* host_mean_speed, float* host_m2_speed, float* host_max_speed,
	uint32_t* host_exceed, uint64_t* samples);
int luw_wind_stats_destroy(luw_wind_stats* st);

/* Wind loads on buildings (momentum exchange). The reference's FORCE_FIELD extension (update_force_field, object_force / object_torque) keeps a 12 B-per-cell
 * force field over the whole lattice and sums it with float atomics; here only the solid cells that touch the fluid are visited, per label (building), and
 * every sum has a fixed order (csrc/lbm_wall_loads.cuh has the definitions).
 * periodic_mask: bit a set = axis a (x y z) is periodic; a link whose partner lies across a GLOBAL face of a non-periodic axis does not count.
 * luw_solid_surface: the listed cells of the domain -- owned solid cells ((flags & 0x03) == TYPE_S) with at least one counted link (partner n - c_i not solid) --
 *   as local dense indices in ascending order, enumerated on the device from the device flags. Two calls: *count first (host_cells NULL), then the list
 *   (capacity >= *count, else LUW_ERR_INVALID). Synchronous; meant to run once per case.
 * luw_wall_loads_create: host_cell_index[count] local dense indices (owned, not halo) with host_label[count] < label_count, sorted by (label, index) strictly
 *   increasing; host_ref_points[3*label_count] the reference point r0 of every label (global lattice coordinates, finite); sample_capacity >= 1 samples of
 *   [label_count][6] doubles are kept on the device until drained. The links are classified once, here, from the device flags. count may be 0.
 * luw_wall_loads_accumulate: one sample of the state whose DDFs are read with time step t (the t luw_update_fields would be given for it): per listed cell
 *   F = 2 x the momentum its counted links carry into the wall (the GAUGE force of the fluid on the cell, relative to the reference pressure 1/3, lattice units),
 *   the Welford update of the mean / M2 of F per cell, and per label the sums of F and of M = (r - r0) x F in double ([Fx Fy Fz Mx My Mz]). Stream-ordered on
 *   the domain's stream, no host synchronisation, no luw_update_fields needed; LUW_ERR_INVALID when sample_capacity samples are pending (the host counts them).
 * luw_wall_loads_drain: synchronous; copies the pending samples out in order, host_loads[s][label][6] (NULL: discard them), *samples = their number, and clears them.
 * luw_wall_loads_download_cells: SoA [c*count + k] over the list, mean_F 3*count, m2_F 3*count; any pointer may be NULL; synchronous; *samples = samples since
 *   create / reset.
 * luw_wall_loads_reset: clears the per-cell statistics and discards the pending samples. */
typedef struct luw_wall_loads luw_wall_loads;
int luw_solid_surface(luw_domain* dom, uint32_t periodic_mask, uint64_t capacity, uint64_t* host_cells, uint64_t* count);
int luw_wall_loads_create(luw_domain* dom, uint64_t count, const uint64_t* host_cell_index, const uint32_t* host_label, uint32_t label_count, const double* host_ref_points,
	uint32_t periodic_mask, uint32_t sample_capacity, luw_wall_loads** out);
int luw_wall_loads_accumulate(luw_wall_loads* st, uint64_t t);
int luw_wall_loads_drain(luw_wall_loads* st, double* host_loads, uint64_t* samples);
int luw_wall_loads_download_cells(luw_wall_loads* st, float* host_mean_F, float* host_m2_F, uint64_t* samples);
int luw_wall_loads_reset(luw_wall_loads* st);
int luw_wall_loads_destroy(luw_wall_loads* st);

/* Probe time series. The reference reads the whole u field back per probe output (FX/setup.cpp:4498-4509), after update_fields over the whole lattice
 * (FX/lbm.cpp:348-355); here one kernel reads the DDFs of the listed cells only, and the samples stay on the device until drained (csrc/lbm_probes.cuh).
 * luw_probes_create: host_cell_index[count] = local dense indices (like luw_cellset_create), owned (not halo) and < Nx*Ny*Nz; duplicates allowed, count may be 0;
 *   sample_capacity >= 1 samples of C*count floats are kept on the device, C = 4 (rho ux uy uz) or 5 (and T, LUW_TEMPERATURE domains).
 * luw_probes_sample: the same arguments as luw_update_fields; per listed cell the rho / u (/ T) that luw_update_fields(t, ...) followed by a read of the fields
 *   would give -- the stored fields on domains with LUW_UPDATE_FIELDS and at the cells update_fields leaves alone -- without writing into the lattice.
 *   Stream-ordered on the domain's stream, no host synchronisation; LUW_ERR_INVALID when sample_capacity samples are pending (the host counts them).
 * luw_probes_drain: synchronous; copies the pending samples out in order, host_values[s][c][k] (NULL: discard them), *samples = their number, and clears them.
 * luw_probes_reset: discards the pending samples. Without a CUDA device every entry returns LUW_ERR_NO_DEVICE. */
typedef struct luw_probes luw_probes;
int luw_probes_create(luw_domain* dom, uint64_t count, const uint64_t* host_cell_index, uint32_t sample_capacity, luw_probes** out);
int luw_probes_sample(luw_probes* pr, uint64_t t, float fx, float fy, float fz, float omega_x, float omega_y, float omega_z);
int luw_probes_drain(luw_probes* pr, float* host_values, uint64_t* samples);
int luw_probes_reset(luw_probes* pr);
int luw_probes_destroy(luw_probes* pr);

/* page-locked host memory for the mirrors (the reference's Memory<T> owns pageable new[] buffers, FX/opencl.hpp:354) */
int luw_host_alloc(void** host_ptr, uint64_t bytes);
int luw_host_free(void* host_ptr);

/* Device::finish_queue, FX/opencl.hpp:323 */
int luw_sync(luw_domain* dom);

/* timing helper for harnesses: CUDA events recorded on the domain's stream around whatever is enqueued between begin and end */
int luw_timer_begin(luw_domain* dom);
int luw_timer_end(luw_domain* dom, float* milliseconds); /* synchronises on the end event */
/* per-kernel timing for harnesses: when enabled, every stream_collide enqueue is bracketed by CUDA events on the domain's stream
 * (the step is a single kernel); luw_kernel_timing_read synchronises and returns the summed duration and the launch count
 * since the last read. */
int luw_kernel_timing(luw_domain* dom, int enable);
int luw_kernel_timing_read(luw_domain* dom, float* milliseconds_total, uint64_t* launches);
/* number of kernels this library has launched on behalf of `dom` since creation */
int luw_launch_count(const luw_domain* dom, uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* LUW_CUDA_H */
