// C ABI of the B200 LBM step (include/luw_cuda.h): domain objects, device memory, stream-ordered copies and kernel enqueues.
// Replaces the Device / Memory<T> / Kernel layer of the reference (FX/opencl.hpp:274-683) for LBM_Domain (FX/lbm.cpp:246-433).
#include "../../include/luw_cuda.h"
#include "lbm_launch.h"
#include "lbm_inlet.cuh"
#include "lbm_wind_stats.cuh"
#include "lbm_wall_loads.cuh"
#include "vox_bins.h"

#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

namespace {

thread_local std::string g_error;

int fail(const int code, const std::string& msg) { g_error = msg; return code; }
int cuda_fail(const cudaError_t e, const char* what) {
	const int code = e==cudaErrorMemoryAllocation ? LUW_ERR_OOM : (e==cudaErrorNoDevice||e==cudaErrorInsufficientDriver||e==cudaErrorInitializationError) ? LUW_ERR_NO_DEVICE : LUW_ERR_CUDA;
	return fail(code, std::string(what)+": "+cudaGetErrorName(e)+" ("+cudaGetErrorString(e)+")");
}
#define CU(call) do { const cudaError_t e_ = (call); if(e_!=cudaSuccess) return cuda_fail(e_, #call); } while(0)

struct DeviceGuard { // every entry point may be called with any current device; restore it on exit
	int prev = -1;
	cudaError_t err;
	explicit DeviceGuard(const int dev) { err = cudaGetDevice(&prev); if(err==cudaSuccess&&prev!=dev) err = cudaSetDevice(dev); }
	~DeviceGuard() { if(prev>=0) cudaSetDevice(prev); }
};

} // namespace

struct luw_domain {
	luw_domain_params p;
	luw::DomainConst c;
	const luw::KernelSet* ks = nullptr;
	cudaStream_t own_stream = nullptr, stream = nullptr;
	cudaStream_t copy_stream = nullptr; // H2D / D2H of cell sets, overlapping the kernels on `stream`
	cudaEvent_t ev0 = nullptr, ev1 = nullptr;
	float* wbuf = nullptr; float* sigma = nullptr;
	uint64_t bytes = 0ull, launches = 0ull;
	uint64_t ncells = 0ull; // Nx*Ny*Nz: cells of the lattice = elements per component of a HOST image (the device arrays have c.N = Px*Ny*Nz, see lbm_common.cuh)
	size_t ddf_size = 4u;
	luw::TileMaps maps; // TMA descriptors for the tiled step
	bool tiled = false; // the tiled step is usable for this domain
	int last_sched_parity = -1; // parity of the last tiled step enqueued (see enqueue_step)
	int tile_variant = 0, sm_count = 0;
	luw::TileShape tile_shape = {}; // box of tile_variant
	struct HaloAxis { // transfer buffers of one decomposed axis (reference: transfer_buffer_p / _m, FX/lbm.cpp:1864-1889) and the events that order their use
		char* send_p = nullptr; char* send_m = nullptr; char* recv_p = nullptr; char* recv_m = nullptr;
		uint64_t bytes = 0ull;
		cudaEvent_t extracted = nullptr, got_p = nullptr, got_m = nullptr; // my payloads are packed / I have copied the (+) and the (-) neighbour's payload out of ITS send buffer
		cudaEvent_t inserted = nullptr; // direct exchange (remote stores into the neighbours' receive buffers): I have unpacked my receive buffers, they may be overwritten
		// (an event can only be recorded on a stream of its own device: every event here is recorded by its owner and waited for by the neighbours)
		bool in_use = false;
	} halo[3];
	struct HaloIpc { // peer-mapped receive block of one axis (luw_halo_ipc_*): [flag_p @0 | flag_m @64 | recv_p[0] recv_m[0] recv_p[1] recv_m[1] @256]
		char* block = nullptr; char* up = nullptr; char* dn = nullptr; // mine, and the mapped blocks of the (+) / (-) neighbour
		uint64_t buf_bytes = 0ull; // one receive buffer, rounded up to 256 B
		uint32_t seq = 0u; // exchanges issued on this axis
		bool same = false; // up and dn are one mapping
	} ipc[3];
	// overlapped halo exchange (luw_step_halo_ipc): second stream, "boundary strips are in global memory" counter of the step kernel and its running target
	cudaStream_t halo_stream = nullptr;
	cudaEvent_t halo_done = nullptr;
	uint32_t bdone_target = 0u;
	uint64_t overlapped_steps = 0ull;
	bool ktiming = false; // bracket every main step kernel with events (luw_kernel_timing)
	std::vector<cudaEvent_t> kev; // event pairs
	size_t kev_used = 0u;
};
struct luw_cellset {
	luw_domain* dom;
	uint64_t count;
	uint64_t* cell; // device: local cell indices
	// Copies run on the domain's copy stream so that they overlap the step kernel; only the small scatter / gather kernels sit on the domain's stream.
	// Two staging slots per direction (4*count bytes per component, up to 3 components), handed round by events:
	float* up[2]; float* dn[2];
	cudaEvent_t staged[2], scattered[2]; // upload: H2D into up[k] finished / the scatter has read up[k]
	cudaEvent_t gathered[2], drained[2]; // download: gather has filled dn[k] / D2H out of dn[k] finished
	uint32_t up_seq, dn_seq;
};
struct luw_stats {
	luw_domain* dom;
	uint64_t count;
	float* mean_u; float* m2_u; float* mean_rho; // device, pitched like u / rho: [c*c.N + n]
	float* mean_T; // LUW_TEMPERATURE domains: running mean of T (avg_T, FX/setup.cpp:4449-4451, 4481-4486); nullptr otherwise
};
struct luw_wind_stats {
	luw_domain* dom;
	uint64_t count, samples;
	uint64_t* cell; // device indices of the listed cells
	float* acc; // [j*count + k], j < luw::WIND_FLOAT_ACCUMULATORS (lbm_wind_stats.cuh)
	uint32_t* exceed; // [j*count + k], j < thr.count
	luw::WindThresholds thr;
};
struct luw_wall_loads {
	luw_domain* dom;
	uint64_t count, nchunks, samples, pending, capacity;
	uint32_t L, periodic;
	uint64_t* cell; // device indices of the listed cells, sorted by (label, index)
	uint32_t* links; // counted links per listed cell (lbm_wall_loads.cuh)
	float* F; // [a*count + k]: the last sample's force per cell
	float* acc; // [a*count + k]: mean of F (a < 3), M2 of F (3 <= a < 6)
	uint64_t* chunk_begin; uint32_t* chunk_label; // [nchunks + 1], [nchunks]: first-level chunks of WALL_CHUNK cells of one label
	uint64_t ngroups;
	uint64_t* group_begin; // [ngroups + 1]: second-level groups of up to WALL_GROUP chunks of one label
	uint64_t* label_group; // [L + 1]: the groups of label l are [label_group[l], label_group[l+1])
	double* ref; // [3L]: reference points
	double* partial; // [a*nchunks + h]
	double* partial2; // [a*ngroups + g]
	double* ring; // [capacity][L][6]: samples not drained yet
};
struct luw_probes {
	luw_domain* dom;
	uint64_t count, pending, capacity;
	uint32_t comps; // 4: rho ux uy uz; 5: and T
	uint64_t* cell; // device indices of the listed cells
	float* ring; // [capacity][comps][count]: samples not drained yet
};
struct luw_vk_inlet {
	luw_domain* dom;
	uint64_t P, M, V;
	uint64_t* point_cell; uint8_t* point_face; float* point_data; float* mode_data;
	float* mode_cs; // [6*V]: A cos(phi), A sin(phi) per component, for the FAST kernel
};

namespace {

int field_info(const luw_domain* d, const int field, void** base, size_t* elem, uint64_t* count) { // count: elements of the dense (host-side) image
	const uint64_t N = d->ncells;
	switch(field) {
		case LUW_FIELD_RHO: *base = d->c.rho; *elem = 4u; *count = N; return LUW_OK;
		case LUW_FIELD_U: *base = d->c.u; *elem = 4u; *count = 3ull*N; return LUW_OK;
		case LUW_FIELD_FLAGS: *base = d->c.flags; *elem = 1u; *count = N; return LUW_OK;
		case LUW_FIELD_FI: *base = d->c.fi; *elem = d->ddf_size; *count = 19ull*N; return LUW_OK;
		case LUW_FIELD_T: if(!d->c.T) return fail(LUW_ERR_INVALID, "field T needs a domain created with LUW_TEMPERATURE"); *base = d->c.T; *elem = 4u; *count = N; return LUW_OK;
		case LUW_FIELD_GI: if(!d->c.gi) return fail(LUW_ERR_INVALID, "field gi needs a domain created with LUW_TEMPERATURE"); *base = d->c.gi; *elem = d->ddf_size; *count = 7ull*N; return LUW_OK;
		default: return fail(LUW_ERR_INVALID, "unknown field id");
	}
}
// device index of the cell with dense index n = x+(y+z*Ny)*Nx
inline uint64_t device_index(const luw::DomainConst& c, const uint64_t n) { return c.Px==c.Nx ? n : (n%c.Nx)+(n/c.Nx)*(uint64_t)c.Px; }
// Copy elements [offset, offset+count) of a dense host image to / from the pitched device array: whole rows with one 2-D copy per component,
// partial rows at the two ends with 1-D copies. With Px == Nx this is the single 1-D copy of the reference (FX/opencl.hpp:481-512).
cudaError_t copy_field(luw_domain* d, char* dev_base, const size_t elem, char* host, const uint64_t offset, const uint64_t count, const bool to_device) {
	const luw::DomainConst& c = d->c;
	const cudaMemcpyKind kind = to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
	if(count==0ull) return cudaSuccess;
	if(c.Px==c.Nx) return to_device ? cudaMemcpyAsync(dev_base+offset*elem, host, count*elem, kind, d->stream) : cudaMemcpyAsync(host, dev_base+offset*elem, count*elem, kind, d->stream);
	const uint64_t N = d->ncells, Nx = c.Nx, Px = c.Px;
	uint64_t i = offset; const uint64_t end = offset+count;
	while(i<end) {
		const uint64_t comp = i/N, n0 = i%N, n1 = (end-comp*N<N) ? end-comp*N : N; // [n0, n1) inside this component
		char* dv = dev_base+comp*c.N*elem;
		char* hs = host+(i-offset)*elem;
		uint64_t n = n0;
		cudaError_t e = cudaSuccess;
		const auto piece = [&](const uint64_t len) { // within one row
			char* dp = dv+device_index(c, n)*elem;
			e = to_device ? cudaMemcpyAsync(dp, hs, len*elem, kind, d->stream) : cudaMemcpyAsync(hs, dp, len*elem, kind, d->stream);
			n += len; hs += len*elem;
		};
		if(n%Nx!=0ull) { const uint64_t len = (Nx-n%Nx<n1-n) ? Nx-n%Nx : n1-n; piece(len); if(e!=cudaSuccess) return e; }
		const uint64_t rows = (n1-n)/Nx;
		if(rows>0ull) {
			char* dp = dv+(n/Nx)*Px*elem;
			e = to_device ? cudaMemcpy2DAsync(dp, Px*elem, hs, Nx*elem, Nx*elem, rows, kind, d->stream) : cudaMemcpy2DAsync(hs, Nx*elem, dp, Px*elem, Nx*elem, rows, kind, d->stream);
			if(e!=cudaSuccess) return e;
			n += rows*Nx; hs += rows*Nx*elem;
		}
		if(n<n1) { piece(n1-n); if(e!=cudaSuccess) return e; }
		i = comp*N+n1;
	}
	return cudaSuccess;
}
uint64_t face_area(const luw::DomainConst& c, const uint32_t axis) {
	return axis==0u ? (uint64_t)c.Ny*c.Nz : axis==1u ? (uint64_t)c.Nz*c.Nx : (uint64_t)c.Nx*c.Ny;
}
template<typename T> int dev_alloc(luw_domain* d, T** ptr, const uint64_t count) {
	const cudaError_t e = cudaMalloc((void**)ptr, count*sizeof(T));
	if(e!=cudaSuccess) { *ptr = nullptr; return cuda_fail(e, "cudaMalloc"); }
	d->bytes += count*sizeof(T);
	return LUW_OK;
}
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
	CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
encode_tiled_fn get_encode_tiled() {
	static encode_tiled_fn fn = nullptr;
	if(!fn) {
		void* p = nullptr;
		cudaDriverEntryPointQueryResult q;
		if(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q)==cudaSuccess&&q==cudaDriverEntryPointSuccess) fn = (encode_tiled_fn)p;
	}
	return fn;
}
// Build the TMA descriptors of a domain for the tile shape of the selected variant (KernelSet::choose_tile). Leaves d->tiled false when the lattice cannot be
// described (row pitch not a multiple of 16 bytes for every array) -- the per-cell kernels are used then.
void setup_tiles(luw_domain* d) {
	d->tiled = false;
	const char* off = getenv("LUW_NO_TILE");
	if(off&&off[0]=='1') return;
	const char* var = getenv("LUW_TILE_VARIANT");
	const luw::DomainConst& c = d->c;
	// odd Nx: the row's last pair holds one cell (rows are padded to Px, a multiple of 16 elements); lbm_tile.cuh `odd_end`
	encode_tiled_fn enc = get_encode_tiled();
	if(!enc) return;
	int want = -1; // the default
	if(var&&var[0]) want = atoi(var)>=0 ? atoi(var) : INT_MAX; // a negative request names no variant: it falls back like any other that is not built
	const int v = d->ks->choose_tile(c.precision, c.features, c.Nx, c.Ny, c.Nz, want, &d->tile_shape);
	if(v<0) return;
	d->tile_variant = v;
	const luw::TileShape& sh = d->tile_shape;
	const cuuint64_t es = d->ddf_size;
	const CUtensorMapDataType dt = es==4u ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16;
	const cuuint64_t dims4[4] = { c.Nx, c.Ny, c.Nz, 19u };
	const cuuint64_t dims4A[4] = { c.Nx, c.Ny, c.Nz, 20u }; // slot 19 does not exist and is never traversed (stride 2 from slot 1 or 2 ends at 17 / 18)
	const cuuint64_t str4[3] = { c.Px*es, (cuuint64_t)c.Px*c.Ny*es, c.N*es }; // rows are Px elements apart (multiples of 16 bytes), boxes are clipped at Nx
	const cuuint32_t box4[4] = { (cuuint32_t)sh.tx, (cuuint32_t)sh.ty, (cuuint32_t)sh.tz, 1u };
	const cuuint32_t box4A[4] = { (cuuint32_t)sh.tx, (cuuint32_t)sh.ty, (cuuint32_t)sh.tz, 18u }; // 9 slots at element stride 2
	const cuuint32_t one4[4] = { 1u, 1u, 1u, 1u };
	const cuuint32_t strideA[4] = { 1u, 1u, 1u, 2u };
	if(enc(&d->maps.fi, dt, 4u, c.fi, dims4, str4, box4, one4,
		CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE)!=CUDA_SUCCESS) return;
	if(enc(&d->maps.fiA, dt, 4u, c.fi, dims4A, str4, box4A, strideA,
		CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE)!=CUDA_SUCCESS) return;
	const cuuint64_t dims3[3] = { c.Nx, c.Ny, c.Nz };
	const cuuint64_t str3[2] = { c.Px, (cuuint64_t)c.Px*c.Ny };
	if(enc(&d->maps.flags, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3u, c.flags, dims3, str3, box4, one4,
		CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE)!=CUDA_SUCCESS) return;
	d->tiled = true;
}
cudaError_t enqueue_step(luw_domain* d, const luw::StepArgs& a, const luw::DomainConst* order = nullptr) { // order: d->c with the so_* strip order of an overlapped halo exchange
	cudaError_t e = cudaSuccess;
	if(d->tiled) { // strip counters of the persistent kernel: step parity p uses sched[p] and zeroes sched[p^1]; a memset is only needed when a parity repeats
		const int par = (int)(a.t&1ull);
		if(par==d->last_sched_parity||d->last_sched_parity<0) { e = cudaMemsetAsync(d->c.sched, 0, 8u, d->stream); if(e!=cudaSuccess) return e; }
		d->last_sched_parity = par;
	}
	if(d->ktiming) { // event pair around the main kernel
		if(d->kev_used+2u>d->kev.size()) for(int k=0; k<2; k++) { cudaEvent_t ev; e = cudaEventCreate(&ev); if(e!=cudaSuccess) return e; d->kev.push_back(ev); }
		e = cudaEventRecord(d->kev[d->kev_used], d->stream); if(e!=cudaSuccess) return e;
	}
	// thermal domains: momentum in the tiled kernel (which leaves the pre-force velocity in c.upre) + the TEMPERATURE block as a second kernel -- unless the buoyancy
	// term is live (f != 0 and beta != 0: the momentum step then depends on this step's T), which takes the fused one-cell-per-thread kernel
	const bool thermal = (d->c.features&luw::F_TEMPERATURE)!=0u;
	const bool buoyant = thermal&&d->c.beta!=0.0f&&(a.fx!=0.0f||a.fy!=0.0f||a.fz!=0.0f);
	if(d->tiled&&!buoyant) {
		e = d->ks->stream_collide_tile(order ? *order : d->c, a, d->maps, d->tile_variant, d->sm_count, d->stream);
		if(e==cudaSuccess&&thermal) { e = d->ks->thermal_g(d->c, a, d->stream); d->launches++; }
	}
	else if(thermal) e = d->ks->stream_collide_thermal(d->c, a, d->stream);
	else e = d->ks->stream_collide(d->c, a, d->stream);
	d->launches++;
	if(e!=cudaSuccess) return e;
	if(d->ktiming) { e = cudaEventRecord(d->kev[d->kev_used+1u], d->stream); if(e!=cudaSuccess) return e; d->kev_used += 2u; }
	return e;
}

// scatter / gather between a staging buffer [c*count + k] and a field with `comps` components of stride N
template<typename T> __global__ void __launch_bounds__(256) k_cellset_scatter(T* __restrict__ field, const uint64_t N, const uint32_t comps, const uint64_t count, const uint64_t* __restrict__ cell, const T* __restrict__ stage) {
	const uint64_t k = (uint64_t)blockIdx.x*blockDim.x+threadIdx.x;
	if(k>=count) return;
	const uint64_t n = cell[k];
	for(uint32_t c=0u; c<comps; c++) field[(uint64_t)c*N+n] = stage[(uint64_t)c*count+k];
}
template<typename T> __global__ void __launch_bounds__(256) k_cellset_gather(const T* __restrict__ field, const uint64_t N, const uint32_t comps, const uint64_t count, const uint64_t* __restrict__ cell, T* __restrict__ stage) {
	const uint64_t k = (uint64_t)blockIdx.x*blockDim.x+threadIdx.x;
	if(k>=count) return;
	const uint64_t n = cell[k];
	for(uint32_t c=0u; c<comps; c++) stage[(uint64_t)c*count+k] = field[(uint64_t)c*N+n];
}

// NVLink peer access from `dev` to every other device of the process (once per ordered pair; a pair without P2P falls back to staged copies)
void enable_peer_access(const int dev, const int ndev) {
	static std::vector<char> done;
	if(done.size()<(size_t)ndev*ndev) done.assign((size_t)ndev*ndev, 0);
	for(int other=0; other<ndev; other++) {
		if(other==dev||done[(size_t)dev*ndev+other]) continue;
		done[(size_t)dev*ndev+other] = 1;
		int can = 0;
		if(cudaDeviceCanAccessPeer(&can, dev, other)==cudaSuccess&&can) { if(cudaDeviceEnablePeerAccess(other, 0)!=cudaSuccess) cudaGetLastError(); } // "already enabled" is fine
	}
}

// flags of the IPC halo exchange: sequence numbers written into the neighbours' blocks after the payload (system-scope release) ...
__global__ void k_halo_signal(uint32_t* flag_a, uint32_t* flag_b, const uint32_t value) {
	__threadfence_system(); // the extract kernel before this one (same stream) has completed: its remote stores are ordered before the flags
	asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flag_a), "r"(value) : "memory");
	asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flag_b), "r"(value) : "memory");
}
// ... and awaited by the receiver before its insert kernel. Bounded: a lost neighbour aborts the launch instead of hanging the device.
__global__ void k_halo_wait(const uint32_t* flag_p, const uint32_t* flag_m, const uint32_t value) {
	const long long t0 = clock64();
	for(int k=0; k<2; k++) {
		const uint32_t* f = k==0 ? flag_p : flag_m;
		uint32_t v;
		for(;;) {
			asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
			if((int32_t)(v-value)>=0) break;
			__nanosleep(200u);
			if(clock64()-t0>120000000000ll) __trap(); // ~60 s at 2 GHz: ranks may reach their first exchange seconds apart (host-side case generation)
		}
	}
}
// FX/setup.cpp:4441-4488 per cell, on the device arrays. Products and sums are rounded separately (explicit intrinsics), as in the reference's host build.
__global__ void __launch_bounds__(256) k_stats_accumulate(const uint64_t N, const float inv_n, const float* __restrict__ rho, const float* __restrict__ u,
	float* __restrict__ mean_u, float* __restrict__ m2_u, float* __restrict__ mean_rho) {
	for(uint64_t n=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; n<N; n+=(uint64_t)gridDim.x*blockDim.x) {
#pragma unroll
		for(uint32_t c=0u; c<3u; c++) {
			const float x = u[(uint64_t)c*N+n];
			float mean = mean_u[(uint64_t)c*N+n];
			const float delta = __fadd_rn(x, -mean);
			mean = __fadd_rn(mean, __fmul_rn(delta, inv_n));
			m2_u[(uint64_t)c*N+n] = __fadd_rn(m2_u[(uint64_t)c*N+n], __fmul_rn(delta, __fadd_rn(x, -mean)));
			mean_u[(uint64_t)c*N+n] = mean;
		}
		const float r = mean_rho[n];
		mean_rho[n] = __fadd_rn(r, __fmul_rn(__fadd_rn(rho[n], -r), inv_n));
	}
}
// running mean of one scalar field, the avg_T line of the same loop (FX/setup.cpp:4483-4485): t_avg += (T - t_avg) * inv_n, rounded like the host build
__global__ void __launch_bounds__(256) k_stats_mean(const uint64_t N, const float inv_n, const float* __restrict__ x, float* __restrict__ mean) {
	for(uint64_t n=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; n<N; n+=(uint64_t)gridDim.x*blockDim.x) {
		const float m = mean[n];
		mean[n] = __fadd_rn(m, __fmul_rn(__fadd_rn(x[n], -m), inv_n));
	}
}
__global__ void k_fill_f32(float* p, const uint64_t n, const float v) {
	for(uint64_t i=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; i<n; i+=(uint64_t)gridDim.x*blockDim.x) p[i] = v;
}

} // namespace

// Inflow-sample searches (lbm_inlet.cuh): host buffers in, host buffers out, cells in batches so that the kept-sample table (256 B per cell) stays bounded.
namespace {
struct DeviceBuffers { // released on every exit path
	std::vector<void*> p;
	~DeviceBuffers() { for(void* q : p) cudaFree(q); }
	template<typename T> cudaError_t get(T** out, const uint64_t count) { *out = nullptr; const cudaError_t e = cudaMalloc((void**)out, (count>0ull ? count : 1ull)*sizeof(T)); if(e==cudaSuccess) p.push_back((void*)*out); return e; }
};
constexpr uint64_t kInletBatch = 1ull<<20;
uint64_t g_inlet_launches = 0ull;
} // namespace

extern "C" {

const char* luw_last_error_string(void) { return g_error.c_str(); }

int luw_device_count(int* count) {
	if(!count) return fail(LUW_ERR_INVALID, "count is null");
	*count = 0;
	const cudaError_t e = cudaGetDeviceCount(count);
	if(e!=cudaSuccess) { *count = 0; return cuda_fail(e, "cudaGetDeviceCount"); }
	return LUW_OK;
}
int luw_get_device_info(int device, luw_device_info* info) {
	if(!info) return fail(LUW_ERR_INVALID, "info is null");
	cudaDeviceProp pr;
	CU(cudaGetDeviceProperties(&pr, device));
	memset(info, 0, sizeof(*info));
	strncpy(info->name, pr.name, sizeof(info->name)-1u);
	info->memory_bytes = (uint64_t)pr.totalGlobalMem;
	info->compute_units = (uint32_t)pr.multiProcessorCount;
	int khz = 0;
	cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
	info->clock_mhz = (uint32_t)(khz/1000);
	info->cc_major = (uint32_t)pr.major; info->cc_minor = (uint32_t)pr.minor;
	return LUW_OK;
}

int luw_domain_create(const luw_domain_params* p, luw_domain** out) {
	if(!p||!out) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	if(p->Nx==0u||p->Ny==0u||p->Nz==0u||p->Dx==0u||p->Dy==0u||p->Dz==0u) return fail(LUW_ERR_INVALID, "lattice and domain counts must be positive");
	if((p->Dx>1u&&p->Nx<4u)||(p->Dy>1u&&p->Ny<4u)||(p->Dz>1u&&p->Nz<4u)) return fail(LUW_ERR_INVALID, "a decomposed axis needs at least 2 cells plus 2 halo layers");
	if(p->precision>2u) return fail(LUW_ERR_INVALID, "precision must be LUW_FP32, LUW_FP16S or LUW_FP16C");
	if(p->arith>1u) return fail(LUW_ERR_INVALID, "arith must be LUW_ARITH_STRICT or LUW_ARITH_FAST");
	if(p->Ny>65535u||p->Nz>65535u) return fail(LUW_ERR_INVALID, "Ny and Nz are limited to 65535 by the launch grid");
	const uint64_t Px = ((uint64_t)p->Nx+15ull)&~15ull; // device row pitch
	const uint64_t N = Px*p->Ny*p->Nz; // elements per component on the device
	if(N>0xFFFFFFFFull) return fail(LUW_ERR_INVALID, "more than 2^32-1 cells per domain"); // the reference switches to 64-bit cell indices here (FX/lbm.cpp:631)
	if((p->features&LUW_BUFFER_NUDGING)&&p->buffer_N==0u) return fail(LUW_ERR_INVALID, "buffer_N must be positive with BUFFER_NUDGING");
	if((p->features&LUW_TOP_SPONGE)&&p->sponge_N==0u) return fail(LUW_ERR_INVALID, "sponge_N must be positive with TOP_SPONGE");
	int ndev = 0;
	{ const cudaError_t e = cudaGetDeviceCount(&ndev); if(e!=cudaSuccess||ndev==0) return e!=cudaSuccess ? cuda_fail(e, "cudaGetDeviceCount") : fail(LUW_ERR_NO_DEVICE, "no CUDA device"); }
	if(p->device<0||p->device>=ndev) return fail(LUW_ERR_INVALID, "device ordinal out of range");
	DeviceGuard guard(p->device);
	if(guard.err!=cudaSuccess) return cuda_fail(guard.err, "cudaSetDevice");

	if(p->Dx*p->Dy*p->Dz>1u) enable_peer_access(p->device, ndev);
	luw_domain* d = new(std::nothrow) luw_domain();
	if(!d) return fail(LUW_ERR_OOM, "host allocation failed");
	d->p = *p;
	d->ks = p->arith==LUW_ARITH_STRICT ? &luw::kernels_strict() : &luw::kernels_fast();
	d->ddf_size = p->precision==LUW_FP32 ? 4u : 2u;
	luw::DomainConst& c = d->c;
	memset(&c, 0, sizeof(c));
	c.Nx = p->Nx; c.Ny = p->Ny; c.Nz = p->Nz; c.Px = (uint32_t)Px; c.N = N;
	d->ncells = (uint64_t)p->Nx*p->Ny*p->Nz;
	c.Dx = p->Dx; c.Dy = p->Dy; c.Dz = p->Dz; c.Ox = p->Ox; c.Oy = p->Oy; c.Oz = p->Oz;
	c.Nxg = (p->Nx-2u*(p->Dx>1u))*p->Dx; c.Nyg = (p->Ny-2u*(p->Dy>1u))*p->Dy; c.Nzg = (p->Nz-2u*(p->Dz>1u))*p->Dz; // FX/lbm.cpp:613-627
	c.wx = -p->Ox; c.ex = (int)c.Nxg-1-p->Ox; c.sy = -p->Oy; c.ny = (int)c.Nyg-1-p->Oy; c.tz = (int)c.Nzg-1-p->Oz;
	c.has_w = c.wx>=0&&c.wx<(int)c.Nx; c.has_e = c.ex>=0&&c.ex<(int)c.Nx;
	c.has_s = c.sy>=0&&c.sy<(int)c.Ny; c.has_n = c.ny>=0&&c.ny<(int)c.Ny; c.has_t = c.tz>=0&&c.tz<(int)c.Nz;
	c.w = p->w; c.tau0 = 1.0f/p->w; c.tau0sq = c.tau0*c.tau0; c.precision = (int)p->precision; c.features = p->features;
	c.downstream_face = p->downstream_face;
	c.buffer_N = p->buffer_N; c.buffer_inv_tau = p->buffer_inv_tau; c.nudge_vertical = p->buffer_nudge_vertical;
	c.sponge_N = p->sponge_N;
	c.w_T = 1.0f; c.beta = 0.0f; c.T_avg = 1.0f; // luw_thermal_params

	int rc = LUW_OK;
	cudaError_t e = cudaStreamCreateWithFlags(&d->own_stream, cudaStreamNonBlocking);
	if(e==cudaSuccess) e = cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking);
	if(e==cudaSuccess) e = cudaEventCreate(&d->ev0);
	if(e==cudaSuccess) e = cudaEventCreate(&d->ev1);
	if(e!=cudaSuccess) rc = cuda_fail(e, "stream/event creation");
	d->stream = d->own_stream;
	if(rc==LUW_OK) rc = dev_alloc(d, (uint8_t**)&c.fi, 19ull*N*d->ddf_size);
	if(rc==LUW_OK) rc = dev_alloc(d, &c.rho, N);
	if(rc==LUW_OK) rc = dev_alloc(d, &c.u, 3ull*N);
	if(rc==LUW_OK) rc = dev_alloc(d, &c.flags, N);
	if(rc==LUW_OK) rc = dev_alloc(d, &c.sched, 4u); // [0], [1]: strip counters of the two step parities; [2]: boundary-strip counter of the overlapped halo exchange (c.bdone)
	const bool thermal = (p->features&LUW_TEMPERATURE)!=0u;
	if(rc==LUW_OK&&thermal) rc = dev_alloc(d, (uint8_t**)&c.gi, 7ull*N*d->ddf_size); // gi = Memory<fpxx>(N, 7), T = Memory<float>(N, 1, .., 1.0f): FX/lbm.cpp:322-323
	if(rc==LUW_OK&&thermal) rc = dev_alloc(d, &c.T, N);
	if(rc==LUW_OK&&thermal) rc = dev_alloc(d, &c.upre, 3ull*N); // two-kernel thermal step: the pre-force velocity handed from the momentum kernel to k_thermal_g (+12 B per cell)
	if(rc==LUW_OK) { // Memory<> zero-fills; rho starts at 1 (FX/lbm.cpp:283-288)
		e = cudaMemsetAsync(c.fi, 0, 19ull*N*d->ddf_size, d->stream);
		if(e==cudaSuccess) e = cudaMemsetAsync(c.u, 0, 3ull*N*4ull, d->stream);
		if(e==cudaSuccess) e = cudaMemsetAsync(c.flags, 0, N, d->stream);
		if(e==cudaSuccess) e = cudaMemsetAsync(c.sched, 0, 16u, d->stream);
		if(e==cudaSuccess) { k_fill_f32<<<1184, 256, 0, d->stream>>>(c.rho, N, 1.0f); e = cudaGetLastError(); d->launches++; }
		if(e==cudaSuccess&&thermal) e = cudaMemsetAsync(c.gi, 0, 7ull*N*d->ddf_size, d->stream);
		if(e==cudaSuccess&&thermal) { k_fill_f32<<<1184, 256, 0, d->stream>>>(c.T, N, 1.0f); e = cudaGetLastError(); d->launches++; }
		if(e!=cudaSuccess) rc = cuda_fail(e, "zero-fill");
	}
	if(rc==LUW_OK&&(p->features&LUW_BUFFER_NUDGING)) { // distance -> sin^2 ramp, float arithmetic as written in FX/kernel.cpp:1579-1581
		std::vector<float> t(p->buffer_N+1u);
		for(uint32_t k=0u; k<=p->buffer_N; k++) { const float xi = 1.0f-(float)k/(float)p->buffer_N; float wb = sinf(1.5707963267948966f*xi); wb *= wb; t[k] = wb; }
		rc = dev_alloc(d, &d->wbuf, t.size());
		if(rc==LUW_OK) { e = cudaMemcpyAsync(d->wbuf, t.data(), t.size()*4u, cudaMemcpyHostToDevice, d->stream); if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream); if(e!=cudaSuccess) rc = cuda_fail(e, "upload nudging table"); }
	}
	if(rc==LUW_OK&&(p->features&LUW_TOP_SPONGE)) { // depth -> inv_tau*sin^2 ramp, FX/kernel.cpp:1602-1605
		std::vector<float> t(p->sponge_N);
		const int Ns = (int)p->sponge_N;
		for(int k=0; k<Ns; k++) { const float xi = Ns>1 ? 1.0f-(float)k/(float)(Ns-1) : 1.0f; float sg = sinf(1.5707963267948966f*xi); sg = p->sponge_inv_tau*sg*sg; t[(size_t)k] = sg; }
		rc = dev_alloc(d, &d->sigma, t.size());
		if(rc==LUW_OK) { e = cudaMemcpyAsync(d->sigma, t.data(), t.size()*4u, cudaMemcpyHostToDevice, d->stream); if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream); if(e!=cudaSuccess) rc = cuda_fail(e, "upload sponge table"); }
	}
	c.wbuf = d->wbuf; c.sigma = d->sigma;
	c.bdone = c.sched ? c.sched+2 : nullptr;
	if(rc==LUW_OK) {
		cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, p->device);
		setup_tiles(d);
	}
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_domain_destroy(d); g_error = keep; return rc; }
	*out = d;
	return LUW_OK;
}

int luw_domain_destroy(luw_domain* d) {
	if(!d) return LUW_OK;
	DeviceGuard guard(d->p.device);
	if(d->own_stream) cudaStreamSynchronize(d->own_stream);
	cudaFree(d->c.fi); cudaFree(d->c.rho); cudaFree(d->c.u); cudaFree(d->c.flags); cudaFree(d->c.sched); cudaFree(d->wbuf); cudaFree(d->sigma); cudaFree(d->c.gi); cudaFree(d->c.T); cudaFree(d->c.upre);
	if(d->halo_stream) { cudaStreamSynchronize(d->halo_stream); cudaStreamDestroy(d->halo_stream); }
	if(d->halo_done) cudaEventDestroy(d->halo_done);
	if(d->ev0) cudaEventDestroy(d->ev0);
	if(d->ev1) cudaEventDestroy(d->ev1);
	for(cudaEvent_t ev : d->kev) cudaEventDestroy(ev);
	for(int a=0; a<3; a++) {
		luw_domain::HaloAxis& h = d->halo[a];
		cudaFree(h.send_p); cudaFree(h.send_m); cudaFree(h.recv_p); cudaFree(h.recv_m);
		if(h.extracted) cudaEventDestroy(h.extracted);
		if(h.inserted) cudaEventDestroy(h.inserted);
		if(h.got_p) cudaEventDestroy(h.got_p);
		if(h.got_m) cudaEventDestroy(h.got_m);
	}
	for(int a=0; a<3; a++) {
		luw_domain::HaloIpc& h = d->ipc[a];
		if(h.up) cudaIpcCloseMemHandle(h.up);
		if(h.dn&&!h.same) cudaIpcCloseMemHandle(h.dn);
		cudaFree(h.block);
	}
	if(d->copy_stream) { cudaStreamSynchronize(d->copy_stream); cudaStreamDestroy(d->copy_stream); }
	if(d->own_stream) cudaStreamDestroy(d->own_stream);
	delete d;
	return LUW_OK;
}

int luw_domain_set_stream(luw_domain* d, void* cuda_stream) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	CU(cudaStreamSynchronize(d->stream)); // work already enqueued on the old stream must not be overtaken
	d->stream = cuda_stream ? (cudaStream_t)cuda_stream : d->own_stream;
	return LUW_OK;
}
int luw_domain_bytes(const luw_domain* d, uint64_t* device_bytes) {
	if(!d||!device_bytes) return fail(LUW_ERR_INVALID, "null argument");
	*device_bytes = d->bytes;
	return LUW_OK;
}

int luw_domain_step_kernel(const luw_domain* d, int* tiled) {
	if(!d||!tiled) return fail(LUW_ERR_INVALID, "null argument");
	*tiled = d->tiled ? 1 : 0;
	return LUW_OK;
}

int luw_upload(luw_domain* d, int field, const void* host_src, uint64_t offset, uint64_t count) {
	if(!d||!host_src) return fail(LUW_ERR_INVALID, "null argument");
	void* base; size_t elem; uint64_t total;
	if(const int rc = field_info(d, field, &base, &elem, &total)) return rc;
	if(offset>total||count>total-offset) return fail(LUW_ERR_INVALID, "upload range exceeds the field");
	DeviceGuard guard(d->p.device);
	CU(copy_field(d, (char*)base, elem, (char*)host_src, offset, count, true));
	return LUW_OK;
}
int luw_download(luw_domain* d, int field, void* host_dst, uint64_t offset, uint64_t count) {
	if(!d||!host_dst) return fail(LUW_ERR_INVALID, "null argument");
	void* base; size_t elem; uint64_t total;
	if(const int rc = field_info(d, field, &base, &elem, &total)) return rc;
	if(offset>total||count>total-offset) return fail(LUW_ERR_INVALID, "download range exceeds the field");
	DeviceGuard guard(d->p.device);
	CU(copy_field(d, (char*)base, elem, (char*)host_dst, offset, count, false));
	return LUW_OK;
}
int luw_device_ptr(luw_domain* d, int field, void** dev_ptr) {
	if(!d||!dev_ptr) return fail(LUW_ERR_INVALID, "null argument");
	size_t elem; uint64_t total;
	return field_info(d, field, dev_ptr, &elem, &total);
}

int luw_thermal_params(luw_domain* d, float w_T, float beta, float T_avg) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	if(!(d->c.features&luw::F_TEMPERATURE)) return fail(LUW_ERR_INVALID, "the domain was created without LUW_TEMPERATURE");
	if(!(w_T>0.0f)) return fail(LUW_ERR_INVALID, "w_T = 1/(2 alpha + 1/2) must be positive");
	d->c.w_T = w_T; d->c.beta = beta; d->c.T_avg = T_avg; // kernel parameters of the launches that follow
	return LUW_OK;
}

int luw_initialize(luw_domain* d) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	if(d->c.features&luw::F_TEMPERATURE) CU(d->ks->initialize_thermal(d->c, d->stream));
	else CU(d->ks->initialize(d->c, d->stream));
	d->launches++;
	return LUW_OK;
}
int luw_stream_collide(luw_domain* d, uint64_t t, float fx, float fy, float fz, float ox, float oy, float oz) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	const luw::StepArgs a = { t, fx, fy, fz, ox, oy, oz };
	CU(enqueue_step(d, a));
	return LUW_OK;
}
int luw_update_fields(luw_domain* d, uint64_t t, float fx, float fy, float fz, float ox, float oy, float oz) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	const luw::StepArgs a = { t, fx, fy, fz, ox, oy, oz };
	if(d->c.features&luw::F_TEMPERATURE) CU(d->ks->update_fields_thermal(d->c, a, d->stream));
	else CU(d->ks->update_fields(d->c, a, d->stream));
	d->launches++;
	return LUW_OK;
}
int luw_run_steps(luw_domain* d, uint64_t t0, uint64_t k, float fx, float fy, float fz, float ox, float oy, float oz) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	if(d->c.Dx*d->c.Dy*d->c.Dz!=1u) return fail(LUW_ERR_INVALID, "luw_run_steps is the single-domain fast path; decomposed runs need a halo exchange between steps");
	DeviceGuard guard(d->p.device);
	for(uint64_t s=0ull; s<k; s++) {
		const luw::StepArgs a = { t0+s, fx, fy, fz, ox, oy, oz };
		CU(enqueue_step(d, a));
	}
	return LUW_OK;
}

int luw_halo_bytes(const luw_domain* d, int payload, uint32_t axis, uint64_t* bytes) {
	if(!d||!bytes||axis>2u) return fail(LUW_ERR_INVALID, "bad argument");
	const uint64_t A = face_area(d->c, axis);
	if(payload==LUW_HALO_FI) *bytes = 5ull*A*d->ddf_size; // transfers*sizeof(fpxx), FX/lbm.cpp:1937-1939
	else if(payload==LUW_HALO_RHO_U_FLAGS) *bytes = 17ull*A; // FX/lbm.cpp:1940-1942
	else if(payload==LUW_HALO_GI&&d->c.gi) *bytes = A*d->ddf_size; // one DDF per face cell: get_area*sizeof(fpxx), FX/lbm.cpp communicate_gi
	else if(payload==LUW_HALO_T&&d->c.T) *bytes = 4ull*A;
	else return fail(LUW_ERR_INVALID, "unknown halo payload (gi / T need a domain created with LUW_TEMPERATURE)");
	return LUW_OK;
}
// one extract or insert kernel of any payload on the domain's stream
static cudaError_t halo_kernel(luw_domain* d, const int payload, const uint32_t axis, const uint64_t t, const bool insert, const bool xfast, void* bp, void* bm) {
	switch(payload) {
		case LUW_HALO_FI: return d->ks->halo_fi(d->c, d->c.precision, axis, (uint32_t)(t&1ull), insert, xfast, bp, bm, d->stream);
		case LUW_HALO_RHO_U_FLAGS: return d->ks->halo_rho_u_flags(d->c, axis, insert, xfast, bp, bm, d->stream);
		case LUW_HALO_GI: return d->ks->halo_gi(d->c, d->c.precision, axis, (uint32_t)(t&1ull), insert, xfast, bp, bm, d->stream);
		case LUW_HALO_T: return d->ks->halo_T(d->c, axis, insert, xfast, bp, bm, d->stream);
		default: return cudaErrorInvalidValue;
	}
}
static bool halo_payload_ok(const luw_domain* d, const int payload) {
	return payload==LUW_HALO_FI||payload==LUW_HALO_RHO_U_FLAGS||((payload==LUW_HALO_GI||payload==LUW_HALO_T)&&d->c.gi&&d->c.T);
}
static int halo(luw_domain* d, int payload, uint32_t axis, uint64_t t, void* bp, void* bm, const bool insert) {
	if(!d||!bp||!bm||axis>2u) return fail(LUW_ERR_INVALID, "bad argument");
	const uint32_t D = axis==0u ? d->c.Dx : axis==1u ? d->c.Dy : d->c.Dz;
	if(D<2u) return fail(LUW_ERR_INVALID, "axis is not decomposed: it has no halo layers");
	if(!halo_payload_ok(d, payload)) return fail(LUW_ERR_INVALID, "unknown halo payload (gi / T need a domain created with LUW_TEMPERATURE)");
	DeviceGuard guard(d->p.device);
	CU(halo_kernel(d, payload, axis, t, insert, false, bp, bm));
	d->launches++;
	return LUW_OK;
}
int luw_halo_extract(luw_domain* d, int payload, uint32_t axis, uint64_t t, void* bp, void* bm) { return halo(d, payload, axis, t, bp, bm, false); }
int luw_halo_insert(luw_domain* d, int payload, uint32_t axis, uint64_t t, const void* bp, const void* bm) { return halo(d, payload, axis, t, (void*)bp, (void*)bm, true); }

static int halo_axis_setup(luw_domain* d, const uint32_t axis) { // buffers sized for the larger payload (rho_u_flags: 17 B per face cell >= 5 fpxx for FP16; FP32: 20 B)
	luw_domain::HaloAxis& h = d->halo[axis];
	if(h.send_p) return LUW_OK;
	DeviceGuard guard(d->p.device);
	const uint64_t A = face_area(d->c, axis);
	h.bytes = A*(d->ddf_size==4u ? 20ull : 17ull);
	int rc = dev_alloc(d, &h.send_p, h.bytes);
	if(rc==LUW_OK) rc = dev_alloc(d, &h.send_m, h.bytes);
	if(rc==LUW_OK) rc = dev_alloc(d, &h.recv_p, h.bytes);
	if(rc==LUW_OK) rc = dev_alloc(d, &h.recv_m, h.bytes);
	if(rc!=LUW_OK) return rc;
	CU(cudaEventCreateWithFlags(&h.extracted, cudaEventDisableTiming));
	CU(cudaEventCreateWithFlags(&h.got_p, cudaEventDisableTiming));
	CU(cudaEventCreateWithFlags(&h.got_m, cudaEventDisableTiming));
	CU(cudaEventCreateWithFlags(&h.inserted, cudaEventDisableTiming));
	return LUW_OK;
}
// can a kernel on device `a` store into memory of device `b`? (peer access is switched on by luw_domain_create for every pair that allows it)
static bool peer_stores_ok(const int a, const int b) {
	if(a==b) return true;
	int can = 0;
	if(cudaDeviceCanAccessPeer(&can, a, b)!=cudaSuccess||!can) { cudaGetLastError(); return false; }
	DeviceGuard guard(a);
	const cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
	if(e!=cudaSuccess) cudaGetLastError(); // "already enabled" is the expected answer
	return e==cudaSuccess||e==cudaErrorPeerAccessAlreadyEnabled;
}
int luw_halo_exchange(luw_domain* const* doms, uint32_t count, int payload, uint32_t axis, uint64_t t) {
	if(!doms||count==0u||axis>2u) return fail(LUW_ERR_INVALID, "bad argument");
	const luw::DomainConst& c0 = doms[0]->c;
	if(count!=c0.Dx*c0.Dy*c0.Dz) return fail(LUW_ERR_INVALID, "luw_halo_exchange needs all Dx*Dy*Dz domains of the decomposition");
	const uint32_t D[3] = { c0.Dx, c0.Dy, c0.Dz };
	if(D[axis]<2u) return LUW_OK; // nothing to exchange on an undecomposed axis
	for(uint32_t i=0u; i<count; i++) {
		if(!doms[i]) return fail(LUW_ERR_INVALID, "null domain");
		if(!halo_payload_ok(doms[i], payload)) return fail(LUW_ERR_INVALID, "unknown halo payload (gi / T need domains created with LUW_TEMPERATURE)");
		if(const int rc = halo_axis_setup(doms[i], axis)) return rc;
	}
	uint64_t bytes = 0ull;
	luw_halo_bytes(doms[0], payload, axis, &bytes);
	const uint32_t stride = axis==0u ? 1u : axis==1u ? D[0] : D[0]*D[1];
	const auto neighbour = [&](const uint32_t i, const uint32_t step) { const uint32_t di = (i/stride)%D[axis]; return doms[i-di*stride+((di+step)%D[axis])*stride]; }; // periodic
	// Direct exchange (all neighbour pairs on one device or with peer access; LUW_HALO_DIRECT=0 keeps the staged copies): like the one-process-per-GPU driver's IPC path,
	// the extract kernel of a domain STORES its two payloads straight into the neighbours' receive buffers over NVLink; events -- all domains live in this process --
	// take the place of the flags. No send buffers, no cudaMemcpyPeerAsync.
	static const bool direct_allowed = []{ const char* e = getenv("LUW_HALO_DIRECT"); return !(e&&e[0]=='0'); }();
	bool direct = direct_allowed;
	for(uint32_t i=0u; i<count&&direct; i++) direct = peer_stores_ok(doms[i]->p.device, neighbour(i, 1u)->p.device)&&peer_stores_ok(doms[i]->p.device, neighbour(i, D[axis]-1u)->p.device);
	if(direct) {
		for(uint32_t i=0u; i<count; i++) { // 1. pack into the neighbours' receive buffers, once they have unpacked the previous exchange of this axis
			luw_domain* d = doms[i];
			luw_domain* up = neighbour(i, 1u);
			luw_domain* dn = neighbour(i, D[axis]-1u);
			DeviceGuard guard(d->p.device);
			if(up->halo[axis].in_use) CU(cudaStreamWaitEvent(d->stream, up->halo[axis].inserted, 0));
			if(dn->halo[axis].in_use) CU(cudaStreamWaitEvent(d->stream, dn->halo[axis].inserted, 0));
			CU(halo_kernel(d, payload, axis, t, false, true, up->halo[axis].recv_m, dn->halo[axis].recv_p)); // my + face -> the (+) neighbour's - halo, my - face -> the (-) neighbour's + halo
			d->launches++;
			CU(cudaEventRecord(d->halo[axis].extracted, d->stream));
		}
		for(uint32_t i=0u; i<count; i++) { // 2. unpack what the two neighbours stored
			luw_domain* d = doms[i];
			luw_domain::HaloAxis& h = d->halo[axis];
			DeviceGuard guard(d->p.device);
			CU(cudaStreamWaitEvent(d->stream, neighbour(i, D[axis]-1u)->halo[axis].extracted, 0));
			CU(cudaStreamWaitEvent(d->stream, neighbour(i, 1u)->halo[axis].extracted, 0));
			CU(halo_kernel(d, payload, axis, t, true, true, h.recv_p, h.recv_m));
			d->launches++;
			CU(cudaEventRecord(h.inserted, d->stream));
			h.in_use = true;
		}
		return LUW_OK;
	}
	// 1. every domain packs its two boundary layers (after its neighbours have taken the previous payloads out of the send buffers)
	for(uint32_t i=0u; i<count; i++) {
		luw_domain* d = doms[i];
		luw_domain::HaloAxis& h = d->halo[axis];
		DeviceGuard guard(d->p.device);
		if(h.in_use) { // send_p was read by the (+) neighbour into its - halo (its got_m), send_m by the (-) neighbour (its got_p)
			CU(cudaStreamWaitEvent(d->stream, neighbour(i, 1u)->halo[axis].got_m, 0));
			CU(cudaStreamWaitEvent(d->stream, neighbour(i, D[axis]-1u)->halo[axis].got_p, 0));
		}
		CU(halo_kernel(d, payload, axis, t, false, true, h.send_p, h.send_m));
		d->launches++;
		CU(cudaEventRecord(h.extracted, d->stream));
	}
	// 2. every domain pulls what its neighbours packed for it (peer copies over NVLink on the RECEIVER's stream) and unpacks it into its halo layers
	for(uint32_t i=0u; i<count; i++) {
		luw_domain* d = doms[i];
		luw_domain* up = neighbour(i, 1u); // (+) neighbour
		luw_domain* dn = neighbour(i, D[axis]-1u); // (-) neighbour
		luw_domain::HaloAxis& h = d->halo[axis];
		DeviceGuard guard(d->p.device);
		// what left the (-) neighbour through its + face arrives in my - halo layer, and vice versa
		CU(cudaStreamWaitEvent(d->stream, dn->halo[axis].extracted, 0));
		CU(cudaMemcpyPeerAsync(h.recv_m, d->p.device, dn->halo[axis].send_p, dn->p.device, bytes, d->stream));
		CU(cudaEventRecord(h.got_m, d->stream));
		CU(cudaStreamWaitEvent(d->stream, up->halo[axis].extracted, 0));
		CU(cudaMemcpyPeerAsync(h.recv_p, d->p.device, up->halo[axis].send_m, up->p.device, bytes, d->stream));
		CU(cudaEventRecord(h.got_p, d->stream));
		h.in_use = true;
		CU(halo_kernel(d, payload, axis, t, true, true, h.recv_p, h.recv_m));
		d->launches++;
	}
	return LUW_OK;
}
static int halo_ipc_axis(luw_domain* d, const uint32_t axis, luw_domain::HaloIpc** out) {
	if(!d||axis>2u) return fail(LUW_ERR_INVALID, "bad argument");
	const uint32_t D = axis==0u ? d->c.Dx : axis==1u ? d->c.Dy : d->c.Dz;
	if(D<2u) return fail(LUW_ERR_INVALID, "axis is not decomposed: it has no halo layers");
	*out = &d->ipc[axis];
	return LUW_OK;
}
int luw_halo_ipc_export(luw_domain* d, uint32_t axis, void* handle_out) {
	luw_domain::HaloIpc* h;
	if(const int rc = halo_ipc_axis(d, axis, &h)) return rc;
	if(!handle_out) return fail(LUW_ERR_INVALID, "null handle");
	DeviceGuard guard(d->p.device);
	if(!h->block) {
		const uint64_t A = face_area(d->c, axis);
		h->buf_bytes = (A*(d->ddf_size==4u ? 20ull : 17ull)+255ull)&~255ull; // the larger payload: 5 fpxx or rho_u_flags (17 B) per face cell
		const uint64_t bytes = 256ull+4ull*h->buf_bytes;
		if(const int rc = dev_alloc(d, &h->block, bytes)) return rc;
		CU(cudaMemsetAsync(h->block, 0, bytes, d->stream));
		CU(cudaStreamSynchronize(d->stream));
	}
	cudaIpcMemHandle_t mh;
	CU(cudaIpcGetMemHandle(&mh, h->block));
	static_assert(sizeof(mh)==64, "cudaIpcMemHandle_t is 64 bytes");
	memcpy(handle_out, &mh, sizeof(mh));
	return LUW_OK;
}
int luw_halo_ipc_connect(luw_domain* d, uint32_t axis, const void* handle_up, const void* handle_dn) {
	luw_domain::HaloIpc* h;
	if(const int rc = halo_ipc_axis(d, axis, &h)) return rc;
	if(!handle_up||!handle_dn) return fail(LUW_ERR_INVALID, "null handle");
	if(!h->block) return fail(LUW_ERR_INVALID, "luw_halo_ipc_export must come first");
	if(h->up) return fail(LUW_ERR_INVALID, "axis is already connected");
	DeviceGuard guard(d->p.device);
	cudaIpcMemHandle_t up, dn;
	memcpy(&up, handle_up, sizeof(up)); memcpy(&dn, handle_dn, sizeof(dn));
	CU(cudaIpcOpenMemHandle((void**)&h->up, up, cudaIpcMemLazyEnablePeerAccess));
	h->same = memcmp(&up, &dn, sizeof(up))==0;
	if(h->same) h->dn = h->up;
	else CU(cudaIpcOpenMemHandle((void**)&h->dn, dn, cudaIpcMemLazyEnablePeerAccess));
	return LUW_OK;
}
int luw_halo_ipc_exchange(luw_domain* d, int payload, uint32_t axis, uint64_t t) {
	luw_domain::HaloIpc* h;
	if(const int rc = halo_ipc_axis(d, axis, &h)) return rc;
	if(!h->up||!h->dn) return fail(LUW_ERR_INVALID, "luw_halo_ipc_connect must come first");
	if(!halo_payload_ok(d, payload)) return fail(LUW_ERR_INVALID, "unknown halo payload (gi / T need a domain created with LUW_TEMPERATURE)");
	DeviceGuard guard(d->p.device);
	const uint32_t seq = h->seq++, par = seq&1u;
	const uint64_t bb = h->buf_bytes;
	// my + face goes into the (+) neighbour's recv_m, my - face into the (-) neighbour's recv_p: remote stores of the extract kernel
	char* const to_up = h->up+256ull+(2ull*par+1ull)*bb;
	char* const to_dn = h->dn+256ull+(2ull*par+0ull)*bb;
	CU(halo_kernel(d, payload, axis, t, false, true, to_up, to_dn));
	k_halo_signal<<<1, 1, 0, d->stream>>>((uint32_t*)(h->up+64), (uint32_t*)(h->dn+0), seq+1u); // the (+) neighbour's flag_m, the (-) neighbour's flag_p
	k_halo_wait<<<1, 1, 0, d->stream>>>((const uint32_t*)(h->block+0), (const uint32_t*)(h->block+64), seq+1u);
	CU(cudaGetLastError());
	char* const recv_p = h->block+256ull+(2ull*par+0ull)*bb;
	char* const recv_m = h->block+256ull+(2ull*par+1ull)*bb;
	CU(halo_kernel(d, payload, axis, t, true, true, recv_p, recv_m));
	d->launches += 4ull;
	return LUW_OK;
}
// the step kernel counts finished boundary strips in *ctr (DomainConst::bdone); the halo stream starts its exchange when all of this step's are in. Bounded like k_halo_wait.
__global__ void k_boundary_wait(const uint32_t* ctr, const uint32_t target) {
	const long long t0 = clock64();
	uint32_t v;
	for(;;) {
		asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
		if((int32_t)(v-target)>=0) break;
		__nanosleep(100u);
		if(clock64()-t0>120000000000ll) __trap();
	}
}
// Strip order of an overlapped step (DomainConst::so_*): the tile rows / planes that hold layers 0, 1, N-2, N-1 of the decomposed y / z axes. false: no interior left to overlap with.
static bool halo_strip_order(const luw_domain* d, luw::DomainConst* o, uint32_t* per_strip) {
	if(!d->tiled) return false;
	const luw::DomainConst& c = d->c;
	const luw::TileShape& sh = d->tile_shape;
	const uint32_t TY = (uint32_t)sh.ty, TZ = (uint32_t)sh.tz, Tx = (c.Nx+(uint32_t)sh.tx-1u)/(uint32_t)sh.tx;
	*o = c;
	if(!luw::strip_order_fill(*o, TY, TZ)) return false;
	const bool park = c.Dx==1u&&Tx>=2u; // the periodic-x column of a strip is flushed by one thread per tile row, a strip later: counted too (lbm_tile.cuh)
	*per_strip = 1u+(park ? TY*TZ : 0u);
	return true;
}
int luw_step_halo_ipc(luw_domain* d, uint64_t t, float fx, float fy, float fz, float ox, float oy, float oz) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	const luw::StepArgs a = { t, fx, fy, fz, ox, oy, oz };
	const bool thermal = (d->c.features&luw::F_TEMPERATURE)!=0u;
	luw::DomainConst order;
	uint32_t per_strip = 0u;
	static const bool allowed = []{ const char* e = getenv("LUW_HALO_OVERLAP"); return !(e&&e[0]=='0'); }();
	const bool overlap = allowed&&!thermal&&d->c.Dx==1u&&(d->c.Dy>1u||d->c.Dz>1u)&&halo_strip_order(d, &order, &per_strip);
	if(!overlap) { // x faces involve every strip, thermal domains run the one-cell-per-thread kernel: exchange behind the step, on the domain's stream
		CU(enqueue_step(d, a));
		for(uint32_t axis=0u; axis<3u; axis++) if((axis==0u ? d->c.Dx : axis==1u ? d->c.Dy : d->c.Dz)>1u) { if(const int rc = luw_halo_ipc_exchange(d, LUW_HALO_FI, axis, t)) return rc; }
		if(thermal) for(uint32_t axis=0u; axis<3u; axis++) if((axis==0u ? d->c.Dx : axis==1u ? d->c.Dy : d->c.Dz)>1u) { if(const int rc = luw_halo_ipc_exchange(d, LUW_HALO_GI, axis, t)) return rc; }
		return LUW_OK;
	}
	if(!d->halo_stream) {
		int lo = 0, hi = 0;
		CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
		CU(cudaStreamCreateWithPriority(&d->halo_stream, cudaStreamNonBlocking, hi)); // its small kernels go ahead of the step kernel's remaining CTAs... which are resident anyway: they only need free thread slots
		CU(cudaEventCreateWithFlags(&d->halo_done, cudaEventDisableTiming));
	}
	CU(enqueue_step(d, a, &order)); // boundary strips first, counted in *c.bdone
	d->bdone_target += order.so_nb*per_strip;
	k_boundary_wait<<<1, 1, 0, d->halo_stream>>>(d->c.bdone, d->bdone_target);
	CU(cudaGetLastError());
	d->launches++;
	cudaStream_t const main_stream = d->stream;
	d->stream = d->halo_stream; // the exchange kernels of luw_halo_ipc_exchange go to the halo stream: they run while the interior strips are still being collided
	int rc = LUW_OK;
	for(uint32_t axis=1u; axis<3u&&rc==LUW_OK; axis++) if((axis==1u ? d->c.Dy : d->c.Dz)>1u) rc = luw_halo_ipc_exchange(d, LUW_HALO_FI, axis, t);
	d->stream = main_stream;
	if(rc!=LUW_OK) return rc;
	CU(cudaEventRecord(d->halo_done, d->halo_stream));
	CU(cudaStreamWaitEvent(d->stream, d->halo_done, 0)); // whatever follows on the domain's stream (the next step, copies, statistics) sees the exchanged lattice
	d->overlapped_steps++;
	return LUW_OK;
}
int luw_overlapped_steps(const luw_domain* d, uint64_t* steps) {
	if(!d||!steps) return fail(LUW_ERR_INVALID, "null argument");
	*steps = d->overlapped_steps;
	return LUW_OK;
}
int luw_run_steps_multi(luw_domain* const* doms, uint32_t count, uint64_t t0, uint64_t k, float fx, float fy, float fz, float ox, float oy, float oz) {
	if(!doms||count==0u) return fail(LUW_ERR_INVALID, "bad argument");
	for(uint64_t s=0ull; s<k; s++) {
		for(uint32_t i=0u; i<count; i++) { if(const int rc = luw_stream_collide(doms[i], t0+s, fx, fy, fz, ox, oy, oz)) return rc; }
		for(uint32_t axis=0u; axis<3u; axis++) { if(const int rc = luw_halo_exchange(doms, count, LUW_HALO_FI, axis, t0+s)) return rc; }
		if(doms[0]&&doms[0]->c.gi) for(uint32_t axis=0u; axis<3u; axis++) { if(const int rc = luw_halo_exchange(doms, count, LUW_HALO_GI, axis, t0+s)) return rc; } // communicate_gi follows communicate_fi, FX/lbm.cpp do_time_step
	}
	return LUW_OK;
}

int luw_vk_inlet_create(luw_domain* d, uint64_t P, uint64_t M, uint64_t V, const uint64_t* pc, const uint8_t* pf, const float* pd, const float* md, luw_vk_inlet** out) {
	if(!d||!out||(P>0ull&&(!pc||!pf||!pd))||(V>0ull&&!md)) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	for(uint64_t i=0ull; i<P; i++) if(pc[i]>=d->ncells) return fail(LUW_ERR_INVALID, "inlet point outside the domain");
	std::vector<uint64_t> pcd(pc, pc+P); // device indices of the cells
	for(uint64_t i=0ull; i<P; i++) pcd[i] = device_index(d->c, pc[i]);
	DeviceGuard guard(d->p.device);
	luw_vk_inlet* v = new(std::nothrow) luw_vk_inlet();
	if(!v) return fail(LUW_ERR_OOM, "host allocation failed");
	memset(v, 0, sizeof(*v));
	v->dom = d; v->P = P; v->M = M; v->V = V;
	int rc = LUW_OK;
	if(P>0ull) {
		rc = dev_alloc(d, &v->point_cell, P);
		if(rc==LUW_OK) rc = dev_alloc(d, &v->point_face, P);
		if(rc==LUW_OK) rc = dev_alloc(d, &v->point_data, 7ull*P);
	}
	if(rc==LUW_OK&&V>0ull) rc = dev_alloc(d, &v->mode_data, 10ull*V);
	if(rc==LUW_OK&&V>0ull) rc = dev_alloc(d, &v->mode_cs, 6ull*V);
	std::vector<float> cs(6ull*V);
	for(uint64_t k=0ull; k<V; k++) for(uint32_t c=0u; c<3u; c++) { // amplitude (rows 4..6) times cos / sin of the phase (rows 7..9), in double, rounded once
		const double A = md[(4ull+c)*V+k], ph = md[(7ull+c)*V+k];
		cs[(2ull*c)*V+k] = (float)(A*cos(ph)); cs[(2ull*c+1ull)*V+k] = (float)(A*sin(ph));
	}
	if(rc==LUW_OK) {
		cudaError_t e = cudaSuccess;
		if(P>0ull) {
			e = cudaMemcpyAsync(v->point_cell, pcd.data(), P*8ull, cudaMemcpyHostToDevice, d->stream);
			if(e==cudaSuccess) e = cudaMemcpyAsync(v->point_face, pf, P, cudaMemcpyHostToDevice, d->stream);
			if(e==cudaSuccess) e = cudaMemcpyAsync(v->point_data, pd, 7ull*P*4ull, cudaMemcpyHostToDevice, d->stream);
		}
		if(e==cudaSuccess&&V>0ull) e = cudaMemcpyAsync(v->mode_data, md, 10ull*V*4ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&V>0ull) e = cudaMemcpyAsync(v->mode_cs, cs.data(), 6ull*V*4ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream); // host arrays may be freed by the caller afterwards
		if(e!=cudaSuccess) rc = cuda_fail(e, "upload inlet buffers");
	}
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_vk_inlet_destroy(v); g_error = keep; return rc; }
	*out = v;
	return LUW_OK;
}
int luw_vk_inlet_apply(luw_vk_inlet* v, uint32_t use_interp, float t0, float t1, float alpha) {
	if(!v) return fail(LUW_ERR_INVALID, "null inlet");
	luw_domain* d = v->dom;
	DeviceGuard guard(d->p.device);
	CU(d->ks->vk_inlet_apply(d->c.N, use_interp, t0, t1, alpha, v->P, v->M, v->V, v->point_cell, v->point_face, v->point_data, v->mode_data, v->mode_cs, d->c.u, d->stream));
	if(v->P>0ull) d->launches++;
	return LUW_OK;
}
int luw_vk_inlet_destroy(luw_vk_inlet* v) {
	if(!v) return LUW_OK;
	DeviceGuard guard(v->dom->p.device);
	cudaStreamSynchronize(v->dom->stream);
	cudaFree(v->point_cell); cudaFree(v->point_face); cudaFree(v->point_data); cudaFree(v->mode_data); cudaFree(v->mode_cs);
	delete v;
	return LUW_OK;
}

int luw_voxelize_mesh(luw_domain* d, uint32_t direction, uint8_t flag, const float* p0, const float* p1, const float* p2, uint32_t ntri, const float* bbu) {
	if(!d||!bbu||(ntri>0u&&(!p0||!p1||!p2))||direction>2u) return fail(LUW_ERR_INVALID, "bad argument");
	for(int k=10; k<16; k++) if(bbu[k]!=0.0f) return fail(LUW_ERR_INVALID, "moving geometry (non-zero linear / rotational velocity) is not supported: LUW voxelises resting meshes only");
	if(ntri==0u) return LUW_OK; // run_voxelize_pass returns early, FX/lbm.cpp:505
	DeviceGuard guard(d->p.device);
	// bin grid over the face (vox_bins.h): every block walks only the triangles near its 32 x 4 columns. LUW_VOXELIZE_BINS=0 keeps the all-triangles kernel (A/B, tests).
	const char* env = getenv("LUW_VOXELIZE_BINS");
	luw::VoxBins bins;
	if(!(env&&env[0]=='0')) bins = luw::vox_build_bins(direction, d->c.Nx, d->c.Ny, d->c.Nz, d->c.Ox, d->c.Oy, d->c.Oz, p0, p1, p2, ntri);
	const bool binned = bins.bins0>0u;
	DeviceBuffers mem;
	float* tri = nullptr; uint32_t* bin_start = nullptr; uint32_t* bin_ids = nullptr;
	CU(mem.get(&tri, 9ull*ntri)); // Memory<float3> p0, p1, p2 of FX/lbm.cpp:525-527: live for this call only
	if(binned) { CU(mem.get(&bin_start, (uint64_t)bins.start.size())); CU(mem.get(&bin_ids, (uint64_t)bins.ids.size())); }
	cudaError_t e = cudaMemcpyAsync(tri, p0, 3ull*ntri*4ull, cudaMemcpyHostToDevice, d->stream);
	if(e==cudaSuccess) e = cudaMemcpyAsync(tri+3ull*ntri, p1, 3ull*ntri*4ull, cudaMemcpyHostToDevice, d->stream);
	if(e==cudaSuccess) e = cudaMemcpyAsync(tri+6ull*ntri, p2, 3ull*ntri*4ull, cudaMemcpyHostToDevice, d->stream);
	if(binned) {
		if(e==cudaSuccess) e = cudaMemcpyAsync(bin_start, bins.start.data(), bins.start.size()*4ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&!bins.ids.empty()) e = cudaMemcpyAsync(bin_ids, bins.ids.data(), bins.ids.size()*4ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess) e = luw::kernels_strict().voxelize_binned(d->c, direction, flag, ntri, bbu+1, bins.bins0, bins.bins1, bin_start, bin_ids, tri, tri+3ull*ntri, tri+6ull*ntri, d->stream);
	} else if(e==cudaSuccess) e = luw::kernels_strict().voxelize(d->c, direction, flag, ntri, bbu+1, tri, tri+3ull*ntri, tri+6ull*ntri, d->stream); // always the as-written arithmetic: flags are bit-exact
	if(e==cudaSuccess) { d->launches++; e = cudaStreamSynchronize(d->stream); } // kernel.run() is synchronous in the reference, and the buffers are released on return
	if(e!=cudaSuccess) return cuda_fail(e, "voxelize_mesh");
	return LUW_OK;
}

int luw_inlet_nearest(int device, uint64_t ncells, const float* cell_xyz, uint32_t npts, const float* point_xyz, uint32_t* nearest) {
	if((ncells>0ull&&(!cell_xyz||!nearest))||(npts>0u&&!point_xyz)) return fail(LUW_ERR_INVALID, "null argument");
	if(ncells==0ull) return LUW_OK;
	DeviceGuard guard(device);
	if(guard.err!=cudaSuccess) return cuda_fail(guard.err, "cudaSetDevice");
	DeviceBuffers mem;
	const uint64_t B = ncells<kInletBatch ? ncells : kInletBatch;
	float* dp = nullptr; float* dc = nullptr; uint32_t* dn = nullptr;
	CU(mem.get(&dp, 3ull*npts)); CU(mem.get(&dc, 3ull*B)); CU(mem.get(&dn, B));
	CU(cudaMemcpy(dp, point_xyz, 3ull*npts*sizeof(float), cudaMemcpyHostToDevice));
	for(uint64_t c0=0ull; c0<ncells; c0+=B) {
		const uint64_t n = ncells-c0<B ? ncells-c0 : B;
		for(int k=0; k<3; k++) CU(cudaMemcpy(dc+(uint64_t)k*n, cell_xyz+(uint64_t)k*ncells+c0, n*sizeof(float), cudaMemcpyHostToDevice));
		luw::k_inlet_nearest<<<(unsigned)((n+127ull)/128ull), 128>>>((uint32_t)n, dc, npts, dp, dn);
		CU(cudaGetLastError());
		g_inlet_launches++;
		CU(cudaMemcpy(nearest+c0, dn, n*sizeof(uint32_t), cudaMemcpyDeviceToHost));
	}
	return LUW_OK;
}

int luw_inlet_knn(int device, uint64_t ncells, const float* cell_ab, uint32_t npts, const float* point_ab, uint32_t* kept, uint32_t* used, float* max_r2, int32_t* exact) {
	if((ncells>0ull&&(!cell_ab||!kept||!used||!max_r2||!exact))||(npts>0u&&!point_ab)) return fail(LUW_ERR_INVALID, "null argument");
	if(ncells==0ull) return LUW_OK;
	DeviceGuard guard(device);
	if(guard.err!=cudaSuccess) return cuda_fail(guard.err, "cudaSetDevice");
	DeviceBuffers mem;
	const uint64_t B = ncells<kInletBatch ? ncells : kInletBatch, K = (uint64_t)luw::INLET_KNN_K;
	float2* dp = nullptr; float* dc = nullptr; uint32_t* dk = nullptr; uint32_t* du = nullptr; float* dm = nullptr; int32_t* de = nullptr;
	CU(mem.get(&dp, (uint64_t)npts)); CU(mem.get(&dc, 2ull*B)); CU(mem.get(&dk, K*B)); CU(mem.get(&du, B)); CU(mem.get(&dm, B)); CU(mem.get(&de, B));
	CU(cudaMemcpy(dp, point_ab, 2ull*npts*sizeof(float), cudaMemcpyHostToDevice));
	for(uint64_t c0=0ull; c0<ncells; c0+=B) {
		const uint64_t n = ncells-c0<B ? ncells-c0 : B;
		for(int k=0; k<2; k++) CU(cudaMemcpy(dc+(uint64_t)k*n, cell_ab+(uint64_t)k*ncells+c0, n*sizeof(float), cudaMemcpyHostToDevice));
		CU(cudaMemset(dk, 0, K*n*sizeof(uint32_t))); // slots beyond used[c] read as 0
		luw::k_inlet_knn<<<(unsigned)((n+(uint64_t)luw::INLET_KNN_THREADS-1ull)/(uint64_t)luw::INLET_KNN_THREADS), luw::INLET_KNN_THREADS>>>((uint32_t)n, dc, npts, dp, dk, du, dm, de);
		CU(cudaGetLastError());
		g_inlet_launches++;
		CU(cudaMemcpy(kept+K*c0, dk, K*n*sizeof(uint32_t), cudaMemcpyDeviceToHost));
		CU(cudaMemcpy(used+c0, du, n*sizeof(uint32_t), cudaMemcpyDeviceToHost));
		CU(cudaMemcpy(max_r2+c0, dm, n*sizeof(float), cudaMemcpyDeviceToHost));
		CU(cudaMemcpy(exact+c0, de, n*sizeof(int32_t), cudaMemcpyDeviceToHost));
	}
	return LUW_OK;
}
int luw_inlet_launch_count(uint64_t* launches) {
	if(!launches) return fail(LUW_ERR_INVALID, "null argument");
	*launches = g_inlet_launches;
	return LUW_OK;
}

int luw_cellset_create(luw_domain* d, uint64_t count, const uint64_t* host_cell_index, luw_cellset** out) {
	if(!d||!out||(count>0ull&&!host_cell_index)) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	for(uint64_t k=0ull; k<count; k++) if(host_cell_index[k]>=d->ncells) return fail(LUW_ERR_INVALID, "cell index outside the domain");
	std::vector<uint64_t> cd(host_cell_index, host_cell_index+count); // device indices
	for(uint64_t k=0ull; k<count; k++) cd[k] = device_index(d->c, host_cell_index[k]);
	DeviceGuard guard(d->p.device);
	luw_cellset* s = new(std::nothrow) luw_cellset();
	if(!s) return fail(LUW_ERR_OOM, "host allocation failed");
	memset(s, 0, sizeof(*s));
	s->dom = d; s->count = count;
	int rc = LUW_OK;
	if(count>0ull) {
		rc = dev_alloc(d, &s->cell, count);
		for(int k=0; k<2&&rc==LUW_OK; k++) { rc = dev_alloc(d, &s->up[k], 3ull*count); if(rc==LUW_OK) rc = dev_alloc(d, &s->dn[k], 3ull*count); }
		for(int k=0; k<2&&rc==LUW_OK; k++) {
			cudaError_t e = cudaEventCreateWithFlags(&s->staged[k], cudaEventDisableTiming);
			if(e==cudaSuccess) e = cudaEventCreateWithFlags(&s->scattered[k], cudaEventDisableTiming);
			if(e==cudaSuccess) e = cudaEventCreateWithFlags(&s->gathered[k], cudaEventDisableTiming);
			if(e==cudaSuccess) e = cudaEventCreateWithFlags(&s->drained[k], cudaEventDisableTiming);
			if(e!=cudaSuccess) rc = cuda_fail(e, "cudaEventCreate");
		}
		if(rc==LUW_OK) {
			cudaError_t e = cudaMemcpyAsync(s->cell, cd.data(), count*8ull, cudaMemcpyHostToDevice, d->stream);
			if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream);
			if(e!=cudaSuccess) rc = cuda_fail(e, "upload cell set");
		}
	}
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_cellset_destroy(s); g_error = keep; return rc; }
	*out = s;
	return LUW_OK;
}
static int cellset_move(luw_cellset* s, int field, void* host, const bool up) {
	if(!s||!host) return fail(LUW_ERR_INVALID, "null argument");
	luw_domain* d = s->dom;
	if(field!=LUW_FIELD_RHO&&field!=LUW_FIELD_U&&field!=LUW_FIELD_FLAGS&&!(field==LUW_FIELD_T&&d->c.T)) return fail(LUW_ERR_INVALID, "cell sets move rho, u, flags or (LUW_TEMPERATURE domains) T");
	if(s->count==0ull) return LUW_OK;
	DeviceGuard guard(d->p.device);
	const uint32_t comps = field==LUW_FIELD_U ? 3u : 1u;
	const size_t elem = field==LUW_FIELD_FLAGS ? 1u : 4u;
	const unsigned blocks = (unsigned)((s->count+255ull)/256ull);
	const size_t bytes = comps*s->count*elem;
	if(up) { // copy stream: wait until the slot's last scatter has read it, H2D; domain stream: wait for the copy, scatter
		const uint32_t k = s->up_seq++&1u;
		CU(cudaStreamWaitEvent(d->copy_stream, s->scattered[k], 0));
		CU(cudaMemcpyAsync(s->up[k], host, bytes, cudaMemcpyHostToDevice, d->copy_stream));
		CU(cudaEventRecord(s->staged[k], d->copy_stream));
		CU(cudaStreamWaitEvent(d->stream, s->staged[k], 0));
		if(field==LUW_FIELD_FLAGS) k_cellset_scatter<uint8_t><<<blocks, 256, 0, d->stream>>>(d->c.flags, d->c.N, 1u, s->count, s->cell, (const uint8_t*)s->up[k]);
		else k_cellset_scatter<float><<<blocks, 256, 0, d->stream>>>(field==LUW_FIELD_U ? d->c.u : field==LUW_FIELD_T ? d->c.T : d->c.rho, d->c.N, comps, s->count, s->cell, s->up[k]);
		CU(cudaGetLastError());
		CU(cudaEventRecord(s->scattered[k], d->stream));
	} else { // domain stream: wait until the slot's last D2H has drained it, gather; copy stream: wait for the gather, D2H
		const uint32_t k = s->dn_seq++&1u;
		CU(cudaStreamWaitEvent(d->stream, s->drained[k], 0));
		if(field==LUW_FIELD_FLAGS) k_cellset_gather<uint8_t><<<blocks, 256, 0, d->stream>>>(d->c.flags, d->c.N, 1u, s->count, s->cell, (uint8_t*)s->dn[k]);
		else k_cellset_gather<float><<<blocks, 256, 0, d->stream>>>(field==LUW_FIELD_U ? d->c.u : field==LUW_FIELD_T ? d->c.T : d->c.rho, d->c.N, comps, s->count, s->cell, s->dn[k]);
		CU(cudaGetLastError());
		CU(cudaEventRecord(s->gathered[k], d->stream));
		CU(cudaStreamWaitEvent(d->copy_stream, s->gathered[k], 0));
		CU(cudaMemcpyAsync(host, s->dn[k], bytes, cudaMemcpyDeviceToHost, d->copy_stream));
		CU(cudaEventRecord(s->drained[k], d->copy_stream));
	}
	d->launches++;
	return LUW_OK;
}
int luw_cellset_upload(luw_cellset* s, int field, const void* host_values) { return cellset_move(s, field, (void*)host_values, true); }
int luw_cellset_download(luw_cellset* s, int field, void* host_values) { return cellset_move(s, field, host_values, false); }
int luw_cellset_destroy(luw_cellset* s) {
	if(!s) return LUW_OK;
	DeviceGuard guard(s->dom->p.device);
	cudaStreamSynchronize(s->dom->stream); cudaStreamSynchronize(s->dom->copy_stream);
	cudaFree(s->cell);
	for(int k=0; k<2; k++) {
		cudaFree(s->up[k]); cudaFree(s->dn[k]);
		if(s->staged[k]) cudaEventDestroy(s->staged[k]);
		if(s->scattered[k]) cudaEventDestroy(s->scattered[k]);
		if(s->gathered[k]) cudaEventDestroy(s->gathered[k]);
		if(s->drained[k]) cudaEventDestroy(s->drained[k]);
	}
	delete s;
	return LUW_OK;
}

int luw_stats_create(luw_domain* d, luw_stats** out) {
	if(!d||!out) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	DeviceGuard guard(d->p.device);
	luw_stats* st = new(std::nothrow) luw_stats();
	if(!st) return fail(LUW_ERR_OOM, "host allocation failed");
	st->dom = d; st->count = 0ull; st->mean_u = st->m2_u = st->mean_rho = st->mean_T = nullptr;
	int rc = dev_alloc(d, &st->mean_u, 3ull*d->c.N);
	if(rc==LUW_OK) rc = dev_alloc(d, &st->m2_u, 3ull*d->c.N);
	if(rc==LUW_OK) rc = dev_alloc(d, &st->mean_rho, d->c.N);
	if(rc==LUW_OK&&d->c.T) rc = dev_alloc(d, &st->mean_T, d->c.N);
	if(rc==LUW_OK) rc = luw_stats_reset(st);
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_stats_destroy(st); g_error = keep; return rc; }
	*out = st;
	return LUW_OK;
}
int luw_stats_reset(luw_stats* st) {
	if(!st) return fail(LUW_ERR_INVALID, "null statistics object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	CU(cudaMemsetAsync(st->mean_u, 0, 3ull*d->c.N*4ull, d->stream));
	CU(cudaMemsetAsync(st->m2_u, 0, 3ull*d->c.N*4ull, d->stream));
	CU(cudaMemsetAsync(st->mean_rho, 0, d->c.N*4ull, d->stream));
	if(st->mean_T) CU(cudaMemsetAsync(st->mean_T, 0, d->c.N*4ull, d->stream));
	st->count = 0ull;
	return LUW_OK;
}
int luw_stats_accumulate(luw_stats* st) {
	if(!st) return fail(LUW_ERR_INVALID, "null statistics object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	st->count++;
	const float inv_n = 1.0f/(float)st->count;
	k_stats_accumulate<<<(unsigned)(4*d->sm_count>0 ? 8*d->sm_count : 1184), 256, 0, d->stream>>>(d->c.N, inv_n, d->c.rho, d->c.u, st->mean_u, st->m2_u, st->mean_rho);
	CU(cudaGetLastError());
	d->launches++;
	if(st->mean_T) {
		k_stats_mean<<<(unsigned)(4*d->sm_count>0 ? 8*d->sm_count : 1184), 256, 0, d->stream>>>(d->c.N, inv_n, d->c.T, st->mean_T);
		CU(cudaGetLastError());
		d->launches++;
	}
	return LUW_OK;
}
int luw_stats_download_temperature(luw_stats* st, float* host_mean_T) {
	if(!st||!host_mean_T) return fail(LUW_ERR_INVALID, "null argument");
	if(!st->mean_T) return fail(LUW_ERR_INVALID, "the statistics object belongs to a domain without LUW_TEMPERATURE");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	CU(copy_field(d, (char*)st->mean_T, 4u, (char*)host_mean_T, 0ull, d->ncells, false));
	CU(cudaStreamSynchronize(d->stream));
	return LUW_OK;
}
int luw_stats_download(luw_stats* st, float* host_mean_u, float* host_m2_u, float* host_mean_rho, uint64_t* count) {
	if(!st) return fail(LUW_ERR_INVALID, "null statistics object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	if(host_mean_u) CU(copy_field(d, (char*)st->mean_u, 4u, (char*)host_mean_u, 0ull, 3ull*d->ncells, false));
	if(host_m2_u) CU(copy_field(d, (char*)st->m2_u, 4u, (char*)host_m2_u, 0ull, 3ull*d->ncells, false));
	if(host_mean_rho) CU(copy_field(d, (char*)st->mean_rho, 4u, (char*)host_mean_rho, 0ull, d->ncells, false));
	CU(cudaStreamSynchronize(d->stream));
	if(count) *count = st->count;
	return LUW_OK;
}
int luw_stats_destroy(luw_stats* st) {
	if(!st) return LUW_OK;
	DeviceGuard guard(st->dom->p.device);
	cudaStreamSynchronize(st->dom->stream);
	cudaFree(st->mean_u); cudaFree(st->m2_u); cudaFree(st->mean_rho); cudaFree(st->mean_T);
	delete st;
	return LUW_OK;
}

static int require_device() { // entry points that may be reached before any domain exists: no device -> LUW_ERR_NO_DEVICE, whatever the other arguments
	int n = 0;
	const cudaError_t e = cudaGetDeviceCount(&n);
	if(e!=cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
	return n>0 ? LUW_OK : fail(LUW_ERR_NO_DEVICE, "no CUDA device");
}
int luw_column_ground(luw_domain* d, uint32_t* host_ground) {
	if(const int rc = require_device()) return rc;
	if(!d||!host_ground) return fail(LUW_ERR_INVALID, "null argument");
	const luw::DomainConst& c = d->c;
	const uint32_t Hz = c.Dz>1u ? 1u : 0u;
	DeviceGuard guard(d->p.device);
	DeviceBuffers mem;
	uint32_t* g = nullptr;
	CU(mem.get(&g, (uint64_t)c.Nx*c.Ny));
	luw::k_column_ground<<<dim3((c.Nx+255u)/256u, c.Ny), 256, 0, d->stream>>>(c.Nx, c.Px, c.Ny, Hz, c.Nz-Hz, c.Oz, c.flags, g);
	CU(cudaGetLastError());
	d->launches++;
	CU(cudaMemcpyAsync(host_ground, g, (uint64_t)c.Nx*c.Ny*4ull, cudaMemcpyDeviceToHost, d->stream));
	CU(cudaStreamSynchronize(d->stream));
	return LUW_OK;
}
int luw_wind_stats_create(luw_domain* d, uint64_t count, const uint64_t* host_cell_index, uint32_t threshold_count, const float* host_thresholds, luw_wind_stats** out) {
	if(const int rc = require_device()) return rc;
	if(!d||!out||(count>0ull&&!host_cell_index)||(threshold_count>0u&&!host_thresholds)) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	if(threshold_count>luw::WIND_MAX_THRESHOLDS) return fail(LUW_ERR_INVALID, "at most LUW_WIND_MAX_THRESHOLDS thresholds");
	luw::WindThresholds thr;
	memset(&thr, 0, sizeof(thr));
	thr.count = threshold_count;
	for(uint32_t j=0u; j<threshold_count; j++) {
		if(!(host_thresholds[j]>=0.0f)) return fail(LUW_ERR_INVALID, "thresholds must be non-negative numbers");
		thr.t[j] = host_thresholds[j];
	}
	for(uint64_t k=0ull; k<count; k++) if(host_cell_index[k]>=d->ncells) return fail(LUW_ERR_INVALID, "cell index outside the domain");
	std::vector<uint64_t> cd(count);
	for(uint64_t k=0ull; k<count; k++) cd[k] = device_index(d->c, host_cell_index[k]);
	DeviceGuard guard(d->p.device);
	luw_wind_stats* st = new(std::nothrow) luw_wind_stats();
	if(!st) return fail(LUW_ERR_OOM, "host allocation failed");
	memset(st, 0, sizeof(*st));
	st->dom = d; st->count = count; st->thr = thr;
	int rc = LUW_OK;
	if(count>0ull) {
		rc = dev_alloc(d, &st->cell, count);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->acc, (uint64_t)luw::WIND_FLOAT_ACCUMULATORS*count);
		if(rc==LUW_OK&&threshold_count>0u) rc = dev_alloc(d, &st->exceed, (uint64_t)threshold_count*count);
		if(rc==LUW_OK) {
			cudaError_t e = cudaMemcpyAsync(st->cell, cd.data(), count*8ull, cudaMemcpyHostToDevice, d->stream);
			if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream); // the host list may be freed by the caller afterwards
			if(e!=cudaSuccess) rc = cuda_fail(e, "upload cell list");
		}
	}
	if(rc==LUW_OK) rc = luw_wind_stats_reset(st);
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_wind_stats_destroy(st); g_error = keep; return rc; }
	*out = st;
	return LUW_OK;
}
int luw_wind_stats_reset(luw_wind_stats* st) {
	if(!st) return fail(LUW_ERR_INVALID, "null statistics object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	if(st->count>0ull) { // every accumulator starts at 0, the running maximum of the speed included (|u| >= 0)
		CU(cudaMemsetAsync(st->acc, 0, (uint64_t)luw::WIND_FLOAT_ACCUMULATORS*st->count*4ull, d->stream));
		if(st->exceed) CU(cudaMemsetAsync(st->exceed, 0, (uint64_t)st->thr.count*st->count*4ull, d->stream));
	}
	st->samples = 0ull;
	return LUW_OK;
}
int luw_wind_stats_accumulate(luw_wind_stats* st) {
	if(!st) return fail(LUW_ERR_INVALID, "null statistics object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	st->samples++;
	const float inv_n = 1.0f/(float)st->samples;
	if(st->count==0ull) return LUW_OK;
	const uint64_t want = (st->count+255ull)/256ull, cap = d->sm_count>0 ? 8ull*(uint64_t)d->sm_count : 1184ull;
	luw::k_wind_stats_accumulate<<<(unsigned)(want<cap ? want : cap), 256, 0, d->stream>>>(st->count, d->c.N, inv_n, d->c.u, st->cell, st->thr, st->acc, st->exceed);
	CU(cudaGetLastError());
	d->launches++;
	return LUW_OK;
}
int luw_wind_stats_download(luw_wind_stats* st, float* host_mean_u, float* host_comoment, float* host_mean_speed, float* host_m2_speed, float* host_max_speed,
	uint32_t* host_exceed, uint64_t* samples) {
	if(!st) return fail(LUW_ERR_INVALID, "null statistics object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	const uint64_t K = st->count;
	if(K>0ull) {
		const auto get = [&](void* host, const void* dev, const uint64_t bytes) { return host ? cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, d->stream) : cudaSuccess; };
		CU(get(host_mean_u, st->acc, 3ull*K*4ull));
		CU(get(host_comoment, st->acc+3ull*K, 6ull*K*4ull));
		CU(get(host_mean_speed, st->acc+9ull*K, K*4ull));
		CU(get(host_m2_speed, st->acc+10ull*K, K*4ull));
		CU(get(host_max_speed, st->acc+11ull*K, K*4ull));
		if(st->exceed) CU(get(host_exceed, st->exceed, (uint64_t)st->thr.count*K*4ull));
	}
	CU(cudaStreamSynchronize(d->stream));
	if(samples) *samples = st->samples;
	return LUW_OK;
}
int luw_wind_stats_destroy(luw_wind_stats* st) {
	if(!st) return LUW_OK;
	DeviceGuard guard(st->dom->p.device);
	cudaStreamSynchronize(st->dom->stream);
	cudaFree(st->cell); cudaFree(st->acc); cudaFree(st->exceed);
	delete st;
	return LUW_OK;
}

// owned range of a local axis: the halo layer at each end of a decomposed axis belongs to the neighbours
static void owned_range(const uint32_t n, const uint32_t D, uint32_t& lo, uint32_t& hi) { lo = D>1u ? 1u : 0u; hi = n-lo; }
static unsigned list_grid(const luw_domain* d, const uint64_t items) {
	const uint64_t want = (items+255ull)/256ull, cap = d->sm_count>0 ? 8ull*(uint64_t)d->sm_count : 1184ull;
	return (unsigned)(want<1ull ? 1ull : want<cap ? want : cap);
}
int luw_solid_surface(luw_domain* d, uint32_t periodic_mask, uint64_t capacity, uint64_t* host_cells, uint64_t* count) {
	if(const int rc = require_device()) return rc;
	if(!d||!count) return fail(LUW_ERR_INVALID, "null argument");
	const luw::DomainConst& c = d->c;
	uint32_t x0, x1, y0, y1, z0, z1;
	owned_range(c.Nx, c.Dx, x0, x1); owned_range(c.Ny, c.Dy, y0, y1); owned_range(c.Nz, c.Dz, z0, z1);
	const uint64_t rows = (uint64_t)(y1-y0)*(z1-z0);
	DeviceGuard guard(d->p.device);
	DeviceBuffers mem;
	uint32_t* rc_dev = nullptr;
	CU(mem.get(&rc_dev, rows));
	luw::k_surface_rows<<<list_grid(d, rows), 256, 0, d->stream>>>(c, periodic_mask&7u, x0, x1, y0, y1, z0, z1, nullptr, rc_dev, nullptr);
	CU(cudaGetLastError());
	d->launches++;
	std::vector<uint32_t> rc(rows);
	CU(cudaMemcpyAsync(rc.data(), rc_dev, rows*4ull, cudaMemcpyDeviceToHost, d->stream));
	CU(cudaStreamSynchronize(d->stream));
	std::vector<uint64_t> offset(rows);
	uint64_t total = 0ull;
	for(uint64_t r=0ull; r<rows; r++) { offset[r] = total; total += rc[r]; }
	*count = total;
	if(!host_cells) return LUW_OK;
	if(capacity<total) return fail(LUW_ERR_INVALID, "capacity below the number of surface cells (call with host_cells == NULL for the count)");
	if(total==0ull) return LUW_OK;
	uint64_t* off_dev = nullptr; uint64_t* cells_dev = nullptr;
	CU(mem.get(&off_dev, rows));
	CU(mem.get(&cells_dev, total));
	CU(cudaMemcpyAsync(off_dev, offset.data(), rows*8ull, cudaMemcpyHostToDevice, d->stream));
	luw::k_surface_rows<<<list_grid(d, rows), 256, 0, d->stream>>>(c, periodic_mask&7u, x0, x1, y0, y1, z0, z1, off_dev, nullptr, cells_dev);
	CU(cudaGetLastError());
	d->launches++;
	CU(cudaMemcpyAsync(host_cells, cells_dev, total*8ull, cudaMemcpyDeviceToHost, d->stream));
	CU(cudaStreamSynchronize(d->stream));
	return LUW_OK;
}
int luw_wall_loads_create(luw_domain* d, uint64_t count, const uint64_t* host_cell_index, const uint32_t* host_label, uint32_t label_count, const double* host_ref_points,
	uint32_t periodic_mask, uint32_t sample_capacity, luw_wall_loads** out) {
	if(const int rc = require_device()) return rc;
	if(!d||!out||(count>0ull&&(!host_cell_index||!host_label))||!host_ref_points) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	if(label_count==0u) return fail(LUW_ERR_INVALID, "label_count must be at least 1");
	if(sample_capacity==0u) return fail(LUW_ERR_INVALID, "sample_capacity must be at least 1");
	for(uint64_t q=0ull; q<3ull*label_count; q++) if(!std::isfinite(host_ref_points[q])) return fail(LUW_ERR_INVALID, "reference points must be finite");
	const luw::DomainConst& c = d->c;
	uint32_t x0, x1, y0, y1, z0, z1;
	owned_range(c.Nx, c.Dx, x0, x1); owned_range(c.Ny, c.Dy, y0, y1); owned_range(c.Nz, c.Dz, z0, z1);
	std::vector<uint64_t> cd(count), chunk_begin;
	std::vector<uint32_t> chunk_label;
	std::vector<uint64_t> label_group(label_count+1ull, 0ull);
	for(uint64_t k=0ull; k<count; k++) {
		const uint64_t n = host_cell_index[k];
		const uint32_t l = host_label[k];
		if(n>=d->ncells) return fail(LUW_ERR_INVALID, "cell index outside the domain");
		const uint32_t x = (uint32_t)(n%c.Nx), y = (uint32_t)((n/c.Nx)%c.Ny), z = (uint32_t)(n/((uint64_t)c.Nx*c.Ny));
		if(x<x0||x>=x1||y<y0||y>=y1||z<z0||z>=z1) return fail(LUW_ERR_INVALID, "cell index in a halo layer");
		if(l>=label_count) return fail(LUW_ERR_INVALID, "label outside [0, label_count)");
		if(k>0ull&&!(l>host_label[k-1ull]||(l==host_label[k-1ull]&&n>host_cell_index[k-1ull]))) return fail(LUW_ERR_INVALID, "the list must be sorted by (label, cell index), strictly increasing");
		if(k==0ull||l!=host_label[k-1ull]||k-chunk_begin.back()==(uint64_t)luw::WALL_CHUNK) { chunk_begin.push_back(k); chunk_label.push_back(l); }
		cd[k] = device_index(c, n);
	}
	const uint64_t nchunks = chunk_label.size();
	chunk_begin.push_back(count);
	std::vector<uint64_t> group_begin;
	for(uint64_t h=0ull; h<nchunks; h++) if(h==0ull||chunk_label[h]!=chunk_label[h-1ull]||h-group_begin.back()==(uint64_t)luw::WALL_GROUP) {
		group_begin.push_back(h);
		label_group[chunk_label[h]+1ull] = group_begin.size(); // label l's groups: [label_group[l], label_group[l+1])
	} else {
		label_group[chunk_label[h]+1ull] = group_begin.size();
	}
	const uint64_t ngroups = group_begin.size();
	group_begin.push_back(nchunks);
	for(uint32_t l=1u; l<=label_count; l++) if(label_group[l]<label_group[l-1u]) label_group[l] = label_group[l-1u]; // labels without cells: empty ranges
	DeviceGuard guard(d->p.device);
	luw_wall_loads* st = new(std::nothrow) luw_wall_loads();
	if(!st) return fail(LUW_ERR_OOM, "host allocation failed");
	memset(st, 0, sizeof(*st));
	st->dom = d; st->count = count; st->nchunks = nchunks; st->ngroups = ngroups; st->L = label_count; st->capacity = sample_capacity; st->periodic = periodic_mask&7u;
	int rc = dev_alloc(d, &st->ref, 3ull*label_count);
	if(rc==LUW_OK) rc = dev_alloc(d, &st->label_group, label_count+1ull);
	if(rc==LUW_OK) rc = dev_alloc(d, &st->ring, (uint64_t)sample_capacity*label_count*luw::WALL_COMPONENTS);
	if(rc==LUW_OK&&count>0ull) {
		rc = dev_alloc(d, &st->cell, count);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->links, count);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->F, 3ull*count);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->acc, 6ull*count);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->chunk_begin, nchunks+1ull);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->chunk_label, nchunks);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->partial, luw::WALL_COMPONENTS*nchunks);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->group_begin, ngroups+1ull);
		if(rc==LUW_OK) rc = dev_alloc(d, &st->partial2, luw::WALL_COMPONENTS*ngroups);
	}
	if(rc==LUW_OK) {
		cudaError_t e = cudaMemcpyAsync(st->ref, host_ref_points, 3ull*label_count*8ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess) e = cudaMemcpyAsync(st->label_group, label_group.data(), (label_count+1ull)*8ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&count>0ull) e = cudaMemcpyAsync(st->group_begin, group_begin.data(), (ngroups+1ull)*8ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&count>0ull) e = cudaMemcpyAsync(st->cell, cd.data(), count*8ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&count>0ull) e = cudaMemcpyAsync(st->chunk_begin, chunk_begin.data(), (nchunks+1ull)*8ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&count>0ull) e = cudaMemcpyAsync(st->chunk_label, chunk_label.data(), nchunks*4ull, cudaMemcpyHostToDevice, d->stream);
		if(e==cudaSuccess&&count>0ull) { // the links are classified once, from the device flags as they are now
			luw::k_wall_links<<<list_grid(d, count), 256, 0, d->stream>>>(c, st->periodic, count, st->cell, st->links);
			e = cudaGetLastError();
			d->launches++;
		}
		if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream); // the host arrays may be freed by the caller afterwards
		if(e!=cudaSuccess) rc = cuda_fail(e, "set up the wall-load list");
	}
	if(rc==LUW_OK) rc = luw_wall_loads_reset(st);
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_wall_loads_destroy(st); g_error = keep; return rc; }
	*out = st;
	return LUW_OK;
}
int luw_wall_loads_reset(luw_wall_loads* st) {
	if(!st) return fail(LUW_ERR_INVALID, "null wall-loads object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	if(st->count>0ull) CU(cudaMemsetAsync(st->acc, 0, 6ull*st->count*4ull, d->stream));
	st->samples = 0ull;
	st->pending = 0ull;
	return LUW_OK;
}
int luw_wall_loads_accumulate(luw_wall_loads* st, uint64_t t) {
	if(!st) return fail(LUW_ERR_INVALID, "null wall-loads object");
	if(st->pending>=st->capacity) return fail(LUW_ERR_INVALID, "the sample ring is full: drain it first");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	const float inv_n = 1.0f/(float)(st->samples+1ull);
	const uint32_t odd = (uint32_t)(t&1ull);
	if(st->count>0ull) {
		const unsigned g = list_grid(d, st->count);
		luw::with_precision(d->c.precision, [&](auto p) { luw::k_wall_cells<decltype(p)::value><<<g, 256, 0, d->stream>>>(d->c, st->count, st->cell, st->links, odd, inv_n, st->F, st->acc); });
		CU(cudaGetLastError());
		luw::k_wall_chunks<<<list_grid(d, st->nchunks), 256, 0, d->stream>>>(d->c, st->count, st->nchunks, st->chunk_begin, st->chunk_label, st->cell, st->F, st->ref, st->partial);
		CU(cudaGetLastError());
		luw::k_wall_segments<<<list_grid(d, st->ngroups*luw::WALL_COMPONENTS), 256, 0, d->stream>>>(st->ngroups, st->group_begin, st->nchunks, st->partial, 1ull, st->ngroups, st->partial2);
		CU(cudaGetLastError());
		d->launches += 3ull;
	}
	luw::k_wall_segments<<<list_grid(d, (uint64_t)st->L*luw::WALL_COMPONENTS), 256, 0, d->stream>>>(st->L, st->label_group, st->ngroups, st->partial2, luw::WALL_COMPONENTS, 1ull,
		st->ring+st->pending*st->L*luw::WALL_COMPONENTS);
	CU(cudaGetLastError());
	d->launches++;
	st->samples++;
	st->pending++;
	return LUW_OK;
}
int luw_wall_loads_drain(luw_wall_loads* st, double* host_loads, uint64_t* samples) {
	if(!st) return fail(LUW_ERR_INVALID, "null wall-loads object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	if(host_loads&&st->pending>0ull) CU(cudaMemcpyAsync(host_loads, st->ring, st->pending*st->L*luw::WALL_COMPONENTS*8ull, cudaMemcpyDeviceToHost, d->stream));
	CU(cudaStreamSynchronize(d->stream));
	if(samples) *samples = st->pending;
	st->pending = 0ull;
	return LUW_OK;
}
int luw_wall_loads_download_cells(luw_wall_loads* st, float* host_mean_F, float* host_m2_F, uint64_t* samples) {
	if(!st) return fail(LUW_ERR_INVALID, "null wall-loads object");
	luw_domain* d = st->dom;
	DeviceGuard guard(d->p.device);
	const uint64_t K = st->count;
	if(K>0ull) {
		if(host_mean_F) CU(cudaMemcpyAsync(host_mean_F, st->acc, 3ull*K*4ull, cudaMemcpyDeviceToHost, d->stream));
		if(host_m2_F) CU(cudaMemcpyAsync(host_m2_F, st->acc+3ull*K, 3ull*K*4ull, cudaMemcpyDeviceToHost, d->stream));
	}
	CU(cudaStreamSynchronize(d->stream));
	if(samples) *samples = st->samples;
	return LUW_OK;
}
int luw_wall_loads_destroy(luw_wall_loads* st) {
	if(!st) return LUW_OK;
	DeviceGuard guard(st->dom->p.device);
	cudaStreamSynchronize(st->dom->stream);
	cudaFree(st->cell); cudaFree(st->links); cudaFree(st->F); cudaFree(st->acc); cudaFree(st->chunk_begin); cudaFree(st->chunk_label);
	cudaFree(st->group_begin); cudaFree(st->label_group); cudaFree(st->ref); cudaFree(st->partial); cudaFree(st->partial2); cudaFree(st->ring);
	delete st;
	return LUW_OK;
}

int luw_probes_create(luw_domain* d, uint64_t count, const uint64_t* host_cell_index, uint32_t sample_capacity, luw_probes** out) {
	if(const int rc = require_device()) return rc;
	if(!d||!out||(count>0ull&&!host_cell_index)) return fail(LUW_ERR_INVALID, "null argument");
	*out = nullptr;
	if(sample_capacity==0u) return fail(LUW_ERR_INVALID, "sample_capacity must be at least 1");
	const luw::DomainConst& c = d->c;
	uint32_t x0, x1, y0, y1, z0, z1;
	owned_range(c.Nx, c.Dx, x0, x1); owned_range(c.Ny, c.Dy, y0, y1); owned_range(c.Nz, c.Dz, z0, z1);
	std::vector<uint64_t> cd(count);
	for(uint64_t k=0ull; k<count; k++) {
		const uint64_t n = host_cell_index[k];
		if(n>=d->ncells) return fail(LUW_ERR_INVALID, "cell index outside the domain");
		const uint32_t x = (uint32_t)(n%c.Nx), y = (uint32_t)((n/c.Nx)%c.Ny), z = (uint32_t)(n/((uint64_t)c.Nx*c.Ny));
		if(x<x0||x>=x1||y<y0||y>=y1||z<z0||z>=z1) return fail(LUW_ERR_INVALID, "cell index in a halo layer");
		cd[k] = device_index(c, n);
	}
	DeviceGuard guard(d->p.device);
	luw_probes* pr = new(std::nothrow) luw_probes();
	if(!pr) return fail(LUW_ERR_OOM, "host allocation failed");
	memset(pr, 0, sizeof(*pr));
	pr->dom = d; pr->count = count; pr->capacity = sample_capacity; pr->comps = (c.features&luw::F_TEMPERATURE) ? 5u : 4u;
	int rc = LUW_OK;
	if(count>0ull) {
		rc = dev_alloc(d, &pr->cell, count);
		if(rc==LUW_OK) rc = dev_alloc(d, &pr->ring, (uint64_t)sample_capacity*pr->comps*count);
		if(rc==LUW_OK) {
			cudaError_t e = cudaMemcpyAsync(pr->cell, cd.data(), count*8ull, cudaMemcpyHostToDevice, d->stream);
			if(e==cudaSuccess) e = cudaStreamSynchronize(d->stream); // cd is freed on return
			if(e!=cudaSuccess) rc = cuda_fail(e, "upload the probe list");
		}
	}
	if(rc!=LUW_OK) { const std::string keep = g_error; luw_probes_destroy(pr); g_error = keep; return rc; }
	*out = pr;
	return LUW_OK;
}
int luw_probes_sample(luw_probes* pr, uint64_t t, float fx, float fy, float fz, float ox, float oy, float oz) {
	if(const int rc = require_device()) return rc;
	if(!pr) return fail(LUW_ERR_INVALID, "null probes object");
	if(pr->pending>=pr->capacity) return fail(LUW_ERR_INVALID, "the sample ring is full: drain it first");
	luw_domain* d = pr->dom;
	if(pr->count>0ull) {
		DeviceGuard guard(d->p.device);
		const luw::StepArgs a = { t, fx, fy, fz, ox, oy, oz };
		CU(d->ks->probe_sample(d->c, a, pr->count, pr->cell, pr->ring+pr->pending*pr->comps*pr->count, list_grid(d, pr->count), d->stream));
		d->launches++;
	}
	pr->pending++;
	return LUW_OK;
}
int luw_probes_drain(luw_probes* pr, float* host_values, uint64_t* samples) {
	if(const int rc = require_device()) return rc;
	if(!pr) return fail(LUW_ERR_INVALID, "null probes object");
	luw_domain* d = pr->dom;
	DeviceGuard guard(d->p.device);
	if(host_values&&pr->pending>0ull&&pr->count>0ull) CU(cudaMemcpyAsync(host_values, pr->ring, pr->pending*pr->comps*pr->count*4ull, cudaMemcpyDeviceToHost, d->stream));
	CU(cudaStreamSynchronize(d->stream));
	if(samples) *samples = pr->pending;
	pr->pending = 0ull;
	return LUW_OK;
}
int luw_probes_reset(luw_probes* pr) {
	if(const int rc = require_device()) return rc;
	if(!pr) return fail(LUW_ERR_INVALID, "null probes object");
	pr->pending = 0ull;
	return LUW_OK;
}
int luw_probes_destroy(luw_probes* pr) {
	if(const int rc = require_device()) return rc;
	if(!pr) return LUW_OK;
	DeviceGuard guard(pr->dom->p.device);
	cudaStreamSynchronize(pr->dom->stream);
	cudaFree(pr->cell); cudaFree(pr->ring);
	delete pr;
	return LUW_OK;
}

int luw_host_alloc(void** host_ptr, uint64_t bytes) {
	if(!host_ptr) return fail(LUW_ERR_INVALID, "null argument");
	*host_ptr = nullptr;
	CU(cudaHostAlloc(host_ptr, bytes, cudaHostAllocPortable));
	return LUW_OK;
}
int luw_host_free(void* host_ptr) {
	if(!host_ptr) return LUW_OK;
	CU(cudaFreeHost(host_ptr));
	return LUW_OK;
}

int luw_sync(luw_domain* d) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	CU(cudaStreamSynchronize(d->stream));
	CU(cudaStreamSynchronize(d->copy_stream)); // cell-set read-backs finish on the copy stream
	return LUW_OK;
}
int luw_timer_begin(luw_domain* d) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	CU(cudaEventRecord(d->ev0, d->stream));
	return LUW_OK;
}
int luw_timer_end(luw_domain* d, float* ms) {
	if(!d||!ms) return fail(LUW_ERR_INVALID, "null argument");
	DeviceGuard guard(d->p.device);
	CU(cudaEventRecord(d->ev1, d->stream));
	CU(cudaEventSynchronize(d->ev1));
	CU(cudaEventElapsedTime(ms, d->ev0, d->ev1));
	return LUW_OK;
}
int luw_kernel_timing(luw_domain* d, int enable) {
	if(!d) return fail(LUW_ERR_INVALID, "null domain");
	DeviceGuard guard(d->p.device);
	CU(cudaStreamSynchronize(d->stream));
	d->ktiming = enable!=0;
	d->kev_used = 0u;
	return LUW_OK;
}
int luw_kernel_timing_read(luw_domain* d, float* ms_total, uint64_t* launches) {
	if(!d||!ms_total||!launches) return fail(LUW_ERR_INVALID, "null argument");
	DeviceGuard guard(d->p.device);
	CU(cudaStreamSynchronize(d->stream));
	float total = 0.0f;
	for(size_t k=0u; k+1u<d->kev_used; k+=2u) { float ms = 0.0f; CU(cudaEventElapsedTime(&ms, d->kev[k], d->kev[k+1u])); total += ms; }
	*ms_total = total; *launches = (uint64_t)(d->kev_used/2u);
	d->kev_used = 0u;
	return LUW_OK;
}
int luw_launch_count(const luw_domain* d, uint64_t* launches) {
	if(!d||!launches) return fail(LUW_ERR_INVALID, "null argument");
	*launches = d->launches;
	return LUW_OK;
}

} // extern "C"
