// C++ host layer of the B200 LBM: the reference's `LBM` / `LBM_Domain` / `Memory<T>` surface (FX/lbm.hpp:26-633, FX/opencl.hpp:331-603) over the
// C ABI of include/luw_cuda.h. FX = core/cfd_core/FluidX3D/src of hweifluids/LatticeUrbanWind.
//
// What is kept (so that FX/setup.cpp, FX/interpolation*.cpp, FX/fluxcorrection.cpp and FX/info.cpp compile against it unchanged):
//   LBM(N, Dx,Dy,Dz, nu, fx,fy,fz, sigma, alpha, beta) and the shorter constructors, run(steps,total), reset(), update_fields(), set_coriolis(),
//   set_fx/fy/fz/f, the getters, coordinates()/index()/position()/center()/size(), lbm.rho / lbm.u / lbm.flags with operator[], .x/.y/.z,
//   length()/dimensions()/range(), read_from_device()/write_to_device(), lbm.lbm_domain[d]-> {rho,u,flags}.enqueue_read_from_device(),
//   finish_queue(), get_Nx()... -- same names, same argument meaning, same error behaviour (print_error -> exit(1), FX/utilities.hpp:4370-4382).
// What is different underneath: no OpenCL, no JIT. The compile-time switches of FX/defines.hpp and the per-case constants the reference bakes
// into the kernel source (FX/lbm.cpp:612-783) are run-time settings (LBM_Settings below; the defaults are LUW's shipped build), the device side is
// the sm_100a library, host mirrors are page-locked, and the halo exchange moves device-to-device (luw_halo_exchange) instead of through the host.
//
// Stand-alone build: this header carries the few types it needs (uint3, float3, ...). Inside the reference tree define LUW_USE_REFERENCE_UTILITIES
// and include FX/utilities.hpp first; the guarded block below then disappears (see INTEGRATION.md).
#pragma once
#include "../../include/luw_cuda.h"

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <chrono>
#include <utility>

#ifndef LUW_USE_REFERENCE_UTILITIES
typedef unsigned int uint;
typedef unsigned char uchar;
typedef uint64_t ulong;
struct uint3 { uint x, y, z; uint3(const uint x=0u, const uint y=0u, const uint z=0u) : x(x), y(y), z(z) {} };
struct float3 { float x, y, z; float3(const float x=0.0f, const float y=0.0f, const float z=0.0f) : x(x), y(y), z(z) {} };
constexpr ulong max_ulong = 18446744073709551615ull;
[[noreturn]] inline void print_error(const std::string& s) { // FX/utilities.hpp:4370-4382: boxed message, then exit(1)
	fprintf(stderr, "+-----------------------------------------------------------------------------+\n| Error: %-68s |\n+-----------------------------------------------------------------------------+\n", s.c_str());
	exit(1);
}
#define TYPE_S 0x01 // FX/defines.hpp:50-57
#define TYPE_E 0x02
#define TYPE_T 0x04
#define TYPE_F 0x08
#define TYPE_I 0x10
#define TYPE_G 0x20
#define TYPE_X 0x40
#define TYPE_Y 0x80
#endif // LUW_USE_REFERENCE_UTILITIES

#ifdef LUW_USE_REFERENCE_UTILITIES // inside the reference tree: the names FX/lbm.hpp:3-21 brings into every translation unit that includes it
#include "defines.hpp" // TYPE_* flag bits, fpxx
#include "units.hpp" // `units` (SI <-> lattice), used by the VTK writer
#include "graphics.hpp" // main_arguments, running (FX/graphics.hpp:16-17; compiles to declarations only when GRAPHICS is off)
#include "info.hpp" // `info` (console progress; FX/info.cpp reads the LBM through the getters below)
#include <fstream>
#include <thread>
extern float3 vtk_origin_shift; // VTK origin shift in SI units (FX/lbm.hpp:10, set by the case driver FX/setup.cpp:4083)
string default_filename(const string& path, const string& name, const string& extension, const ulong t); // FX/lbm.cpp:235-242
string default_filename(const string& name, const string& extension, const ulong t);
uint bytes_per_cell_host(); // FX/lbm.hpp:13-15, for THIS build's buffers and the precision in use
uint bytes_per_cell_device();
uint bandwidth_bytes_per_cell_device();
struct LBM_Device_Info { uint id = 0u; string name = ""; uint memory = 0u, memory_used = 0u; bool uses_ram = false; uint compute_units = 0u, clock_frequency = 0u; }; // the Device_Info fields FX/info.cpp:233-241 prints
struct Device { LBM_Device_Info info; luw_domain* dom = nullptr; }; // what LBM_Domain::get_device() hands out (reference: the OpenCL Device, FX/opencl.hpp:274): its info block + the C-ABI handle
#endif // LUW_USE_REFERENCE_UTILITIES

uint vram_required_mb_per_device(const uint Nx, const uint Ny, const uint Nz, const uint Dx, const uint Dy, const uint Dz); // FX/lbm.hpp:17-18 -- for THIS build's buffers
uint vram_required_mb_total(const uint Nx, const uint Ny, const uint Nz, const uint Dx, const uint Dy, const uint Dz);
// Run-time replacement of FX/defines.hpp + the constants of FX/lbm.cpp:612-783. Set the global `lbm_settings` before constructing an LBM
// (the case driver does that where the reference's update_coriolis / update_buffer_nudging / update_top_sponge set their globals, FX/setup.cpp:3800-3903).
struct LBM_Settings {
	uint precision = LUW_FP16C; // FX/defines.hpp:14 (LUW ships FP16C); LUW_FP32 / LUW_FP16S / LUW_FP16C; env LUW_PRECISION overrides
	uint features = LUW_UPDATE_FIELDS|LUW_VOLUME_FORCE|LUW_EQUILIBRIUM_BOUNDARIES|LUW_SUBGRID; // FX/defines.hpp:17-24; nudging / sponge added by the setters below; |= LUW_TEMPERATURE for the thermal D3Q7 extension (FX/defines.hpp:23; env LUW_TEMPERATURE=1)
	uint arith = LUW_ARITH_FAST; // the reference builds with -cl-mad-enable (FX/opencl.hpp:305); LUW_ARITH_STRICT reproduces the CPU oracle bit for bit
	int downstream_face = 0; // def_downstream_face
	uint buffer_N = 0u; float buffer_inv_tau = 0.0f; int buffer_nudge_vertical = 0; // BUFFER_NUDGING (FX/lbm.cpp:770-776)
	uint sponge_N = 0u; float sponge_inv_tau = 0.0f; // TOP_SPONGE (FX/lbm.cpp:777-782)
	std::vector<int> devices; // CUDA ordinals, one per domain (empty: domain d -> device d % device_count; the reference insists on one card per domain, FX/lbm.cpp:961-979)
	void set_buffer_nudging(const uint N, const float inv_tau, const bool vertical) { buffer_N = N; buffer_inv_tau = inv_tau; buffer_nudge_vertical = vertical ? 1 : 0; if(N>0u) features |= LUW_BUFFER_NUDGING; else features &= ~(uint)LUW_BUFFER_NUDGING; }
	void set_top_sponge(const uint N, const float inv_tau) { sponge_N = N; sponge_inv_tau = inv_tau; if(N>0u) features |= LUW_TOP_SPONGE; else features &= ~(uint)LUW_TOP_SPONGE; }
};
extern LBM_Settings lbm_settings;

float lbm_kernel_literal(const float x); // the float the reference's kernel sees for a constant printed by to_string(float) with 8 decimals (FX/utilities.hpp:2741-2750)
inline void luw_check(const int rc) { if(rc!=LUW_OK) print_error(std::string("CUDA layer: ")+luw_last_error_string()); } // reference: any device error -> print_error (FX/opencl.hpp:613-618)

// ---------------------------------------------------------------------------------------------------------------- Memory<T> (FX/opencl.hpp:331-603)
// Host mirror + the device field of ONE domain. `d` dimensions, SoA: data()[n + c*N].
// The mirror is LAZY: nothing is allocated until the host touches it (data(), operator[], reset, a read from the device). The device field holds the construction
// value from luw_domain_create on, so an untouched mirror has nothing to upload: enqueue_write_to_device() of such a mirror is a no-op. A case that feeds its
// boundary through cell sets (luw_cellset_*) and reads probes the same way therefore never owns a host image of the lattice -- the reference's 17 B per cell of
// host memory (FX/lbm.cpp:95-106; 171 GB for the 10 G-cell configuration) are only paid by code that really indexes the whole field, like the case driver.
// Mirrors up to LUW_PIN_LIMIT_MB (default 4096 MB per field) are page-locked; larger ones are pageable, zero pages committed on first touch.
inline ulong luw_pin_limit_bytes() { static const ulong v = []{ const char* e = getenv("LUW_PIN_LIMIT_MB"); return (ulong)(e ? atol(e) : 4096l)*1048576ull; }(); return v; }
template<typename T> class Memory {
private:
	luw_domain* dom = nullptr;
	int field = 0;
	ulong N = 0ull; uint d = 1u;
	mutable T* host = nullptr;
	mutable bool pinned = false;
	T fill = (T)0; // value of an untouched mirror (= what the device field was created with)
	bool loose = false; // host-only buffer that is not a field of the lattice (see below)
	void release() { if(host) { if(loose) delete[] host; else if(pinned) luw_host_free(host); else free(host); } host = nullptr; x = y = z = nullptr; }
	void materialize() const {
		if(host||N*(ulong)d==0ull) return;
		const ulong bytes = N*(ulong)d*sizeof(T);
		if(bytes<=luw_pin_limit_bytes()) { void* p = nullptr; luw_check(luw_host_alloc(&p, bytes)); host = (T*)p; pinned = true; }
		else { host = (T*)calloc((size_t)(N*(ulong)d), sizeof(T)); pinned = false; if(!host) print_error("Host allocation of "+std::to_string(bytes/1048576ull)+" MB failed."); }
		x = host; if(d>1u) y = host+N; if(d>2u) z = host+2ull*N;
		if(pinned||fill!=(T)0) for(ulong i=0ull; i<N*(ulong)d; i++) host[i] = fill; // calloc'ed zero pages stay uncommitted until they are written
	}
public:
	mutable T* x = nullptr; mutable T* y = nullptr; mutable T* z = nullptr; // host pointers of the components (FX/opencl.hpp:343-349); valid once the mirror has been touched (data())
	Memory() {}
	Memory(luw_domain* dom, const int field, const ulong N, const uint dimensions, const T value) : dom(dom), field(field), N(N), d(dimensions), fill(value) {
		if(N*(ulong)d==0ull) print_error("Memory size must be larger than 0.");
	}
	Memory(const Memory&) = delete;
	Memory& operator=(const Memory&) = delete;
	Memory(Memory&& o) noexcept { *this = std::move(o); }
	Memory& operator=(Memory&& o) noexcept {
		if(this!=&o) { release(); dom = o.dom; field = o.field; N = o.N; d = o.d; host = o.host; pinned = o.pinned; fill = o.fill; loose = o.loose; x = o.x; y = o.y; z = o.z; o.host = nullptr; o.x = o.y = o.z = nullptr; o.N = 0ull; }
		return *this;
	}
	~Memory() { release(); }
#ifdef LUW_USE_REFERENCE_UTILITIES
	// Memory<T>(device, N, dimensions, allocate_host, allocate_device, value, external) of FX/opencl.hpp:383-391 for buffers that are NOT fields of the lattice: the case
	// driver packs the von Karman inlet's point / mode tables into such objects (FX/setup.cpp:1040-1074). Host side only; the Kernel object below takes the contents.
	Memory(Device& device, const ulong N, const uint dimensions=1u, const bool=true, const bool=true, const T value=(T)0, const bool=false) : N(N), d(dimensions), loose(true) {
		(void)device;
		if(N*(ulong)d==0ull) print_error("Memory size must be larger than 0.");
		host = new T[N*(ulong)d];
		x = host; if(d>1u) y = host+N; if(d>2u) z = host+2ull*N;
		reset(value);
	}
#endif
	bool materialized() const { return host!=nullptr; } // has the host ever touched this mirror?
	void reset(const T value=(T)0) { if(!host&&!loose) { fill = value; materialize(); return; } for(ulong i=0ull; i<range(); i++) host[i] = value; }
	ulong length() const { return N; }
	uint dimensions() const { return d; }
	ulong range() const { return N*(ulong)d; }
	ulong capacity() const { return N*(ulong)d*sizeof(T); }
	T* data() { materialize(); return host; }
	const T* data() const { materialize(); return host; }
	T& operator[](const ulong i) { materialize(); return host[i]; }
	const T& operator[](const ulong i) const { materialize(); return host[i]; }
	T operator()(const ulong i) const { materialize(); return host[i]; }
	T operator()(const ulong i, const uint dimension) const { materialize(); return host[i+(ulong)dimension*N]; }
	void enqueue_read_from_device() { if(!loose) { materialize(); luw_check(luw_download(dom, field, host, 0ull, range())); } }
	void enqueue_write_to_device() { if(!loose&&host) luw_check(luw_upload(dom, field, host, 0ull, range())); } // untouched mirror: the device already holds its value
	void enqueue_read_from_device(const ulong offset, const ulong length) { if(!loose) { materialize(); luw_check(luw_download(dom, field, host+offset, offset, length)); } }
	void enqueue_write_to_device(const ulong offset, const ulong length) { if(!loose&&host) luw_check(luw_upload(dom, field, host+offset, offset, length)); }
	void finish_queue() { if(!loose) luw_check(luw_sync(dom)); }
	void read_from_device() { enqueue_read_from_device(); finish_queue(); }
	void write_to_device() { enqueue_write_to_device(); finish_queue(); }
	void read_from_device(const ulong offset, const ulong length) { enqueue_read_from_device(offset, length); finish_queue(); }
	void write_to_device(const ulong offset, const ulong length) { enqueue_write_to_device(offset, length); finish_queue(); }
};

#ifdef LUW_USE_REFERENCE_UTILITIES
// The one Kernel object the case driver creates itself (FX/setup.cpp:1076-1086): Kernel(device, N, "vk_inlet_apply", use_interp, t0, t1, alpha, point_count, mode_count,
// mode_stride, point_cell, point_face, point_data, mode_data, u) and, per step, set_parameters(0u, use_interp, t0, t1, alpha).enqueue_run() (FX/setup.cpp:553).
// Here it owns a luw_vk_inlet built from the packed tables; any other kernel name is an error (there is no OpenCL program behind this layer).
class Kernel {
private:
	luw_vk_inlet* vk = nullptr;
	uint use_interp = 0u; float t0 = 0.0f, t1 = 0.0f, alpha = 0.0f;
public:
	Kernel() {}
	Kernel(const Device& device, const ulong N, const string& name, const uint use_interp, const float t0, const float t1, const float alpha, const ulong point_count, const ulong mode_count, const ulong mode_stride,
		Memory<ulong>& point_cell, Memory<uchar>& point_face, Memory<float>& point_data, Memory<float>& mode_data, Memory<float>& u) : use_interp(use_interp), t0(t0), t1(t1), alpha(alpha) {
		(void)N; (void)u; // the velocity field is the domain's own
		if(name!="vk_inlet_apply") print_error("Kernel \""+name+"\": only vk_inlet_apply can be created by the case driver in this build.");
		static_assert(sizeof(ulong)==sizeof(uint64_t), "point_cell is an array of 64-bit cell indices");
		luw_check(luw_vk_inlet_create(device.dom, point_count, mode_count, mode_stride, (const uint64_t*)point_cell.data(), point_face.data(), point_data.data(), mode_data.data(), &vk));
	}
	Kernel(const Kernel&) = delete;
	Kernel& operator=(const Kernel&) = delete;
	Kernel(Kernel&& o) noexcept { *this = std::move(o); }
	Kernel& operator=(Kernel&& o) noexcept { if(this!=&o) { if(vk) luw_vk_inlet_destroy(vk); vk = o.vk; use_interp = o.use_interp; t0 = o.t0; t1 = o.t1; alpha = o.alpha; o.vk = nullptr; } return *this; }
	~Kernel() { if(vk) luw_vk_inlet_destroy(vk); }
	Kernel& set_parameters(const uint position, const uint use_interp_, const float t0_, const float t1_, const float alpha_) {
		if(position!=0u) print_error("Kernel::set_parameters: vk_inlet_apply takes its per-step arguments from position 0.");
		use_interp = use_interp_; t0 = t0_; t1 = t1_; alpha = alpha_;
		return *this;
	}
	Kernel& enqueue_run() { if(vk) luw_check(luw_vk_inlet_apply(vk, use_interp, t0, t1, alpha)); return *this; }
	Kernel& run() { return enqueue_run(); }
};
#endif // LUW_USE_REFERENCE_UTILITIES

// Per-domain triangle culling of LBM::voxelize_mesh_on_device (FX/lbm.cpp:41-90, 1457-1495): the ids of the triangles whose bounding box, projected along the ray
// direction, overlaps the projected extent [O, O+N-1] of the local lattice (halo layers included), padded by 1 cell + 1e-4. Rays of this domain's columns cannot hit
// any other triangle, so the flags are those of the whole mesh -- except that a domain whose list is EMPTY is skipped altogether by the reference (FX/lbm.cpp:499),
// i.e. previously solid cells inside the mesh's bounding box are not released there. p0/p1/p2: 3 floats per triangle in lattice coordinates.
std::vector<uint> luw_cull_triangles(const float* p0, const float* p1, const float* p2, const uint triangle_number, const uint direction,
	const int Ox, const int Oy, const int Oz, const uint local_Nx, const uint local_Ny, const uint local_Nz);

// ---------------------------------------------------------------------------------------------------------------- LBM_Domain (FX/lbm.hpp:26-221)
// Test hook (tests/test_reference_driver.py): with LUW_DUMP_DIR set, a single-domain LBM writes what it is given and what it computes as raw arrays -- the
// triangles of every voxelisation call, the host images at initialize(), rho / u after step LUW_DUMP_STEP -- so that the deck-driven path through the
// reference's unmodified case driver can be compared with the oracle bit for bit. Never on in production (one getenv at start-up).
bool luw_dump_enabled();
void luw_dump_array(const char* name, const void* data, const ulong bytes);
void luw_dump_voxelize_call(luw_domain* handle, const ulong N, const uint direction, const uchar flag, const float* p0, const float* p1, const float* p2, const uint triangle_number, const float* bbu);

class LBM_Domain {
private:
	uint Nx=1u, Ny=1u, Nz=1u, Dx=1u, Dy=1u, Dz=1u; int Ox=0, Oy=0, Oz=0;
	ulong t = 0ull;
	float nu = 1.0f/6.0f, fx=0.0f, fy=0.0f, fz=0.0f, omega_x=0.0f, omega_y=0.0f, omega_z=0.0f;
	float alpha = 0.0f, beta = 0.0f, T_avg = 1.0f; // thermal diffusion / expansion coefficients, average temperature (FX/lbm.hpp:37)
	int device = 0;
	luw_domain* handle = nullptr; // declared before the buffers: they are built on it
	ulong t_last_update_fields = max_ulong;
	static luw_domain* create_handle(const int device, const uint Nx, const uint Ny, const uint Nz, const uint Dx, const uint Dy, const uint Dz, const int Ox, const int Oy, const int Oz, const float nu, const float alpha, const float beta);
public:
	Memory<float> rho; Memory<float> u; Memory<uchar> flags; // host + device buffers of this domain (FX/lbm.hpp:60-63; rho starts at 1, u and flags at 0: FX/lbm.cpp:283-288)
	Memory<float> T; // temperature (FX/lbm.hpp:77, starts at 1: FX/lbm.cpp:323); only allocated with LUW_TEMPERATURE (length() == 0 otherwise). gi stays device-only like in the reference

	LBM_Domain(const int device, const uint Nx, const uint Ny, const uint Nz, const uint Dx, const uint Dy, const uint Dz, const int Ox, const int Oy, const int Oz,
		const float nu, const float fx, const float fy, const float fz, const float alpha=0.0f, const float beta=0.0f);
	static bool thermal() { return (lbm_features()&LUW_TEMPERATURE)!=0u; }
	float get_alpha() const { return alpha; } float get_beta() const { return beta; } float get_T_avg() const { return T_avg; } // FX/lbm.hpp:151-153
	~LBM_Domain();
	LBM_Domain(const LBM_Domain&) = delete;
	LBM_Domain& operator=(const LBM_Domain&) = delete;

	void enqueue_initialize() { luw_check(luw_initialize(handle)); } // FX/lbm.cpp:340-343
	void enqueue_stream_collide() { luw_check(luw_stream_collide(handle, t, fx, fy, fz, omega_x, omega_y, omega_z)); } // FX/lbm.cpp:344-346
	void enqueue_update_fields() { // FX/lbm.cpp:348-355: only when UPDATE_FIELDS is off, and only once per time step
		if(!(lbm_features()&LUW_UPDATE_FIELDS)&&t!=t_last_update_fields) { luw_check(luw_update_fields(handle, t, fx, fy, fz, omega_x, omega_y, omega_z)); t_last_update_fields = t; }
	}
	void increment_time_step(const uint steps=1u) { t += (ulong)steps; }
	void reset_time_step() { t = 0ull; }
	void finish_queue() { luw_check(luw_sync(handle)); }

	uint get_Nx() const { return Nx; } uint get_Ny() const { return Ny; } uint get_Nz() const { return Nz; }
	ulong get_N() const { return (ulong)Nx*(ulong)Ny*(ulong)Nz; }
	uint get_Dx() const { return Dx; } uint get_Dy() const { return Dy; } uint get_Dz() const { return Dz; }
	uint get_D() const { return Dx*Dy*Dz; }
	int get_Ox() const { return Ox; } int get_Oy() const { return Oy; } int get_Oz() const { return Oz; }
	float get_nu() const { return nu; } float get_fx() const { return fx; } float get_fy() const { return fy; } float get_fz() const { return fz; }
	ulong get_t() const { return t; }
	void set_fx(const float v) { fx = v; } void set_fy(const float v) { fy = v; } void set_fz(const float v) { fz = v; }
	void set_f(const float x, const float y, const float z) { fx = x; fy = y; fz = z; }
	void set_coriolis(const float x, const float y, const float z) { omega_x = x; omega_y = y; omega_z = z; } // FX/lbm.hpp:156-160
	float get_omega_x() const { return omega_x; } float get_omega_y() const { return omega_y; } float get_omega_z() const { return omega_z; } // FX/lbm.hpp:144-146
	uint get_velocity_set() const { return 19u; } // D3Q19, FX/defines.hpp:7
	// LBM_Domain::voxelize_mesh_on_device for TYPE_S geometry (FX/lbm.cpp:494-605: bounding box -+ 2 cells, rays along z unless overridden, resting mesh).
	// p0/p1/p2: 3 floats per triangle in lattice coordinates (Mesh::p0/p1/p2 of FX/utilities.hpp are float3 arrays with exactly this memory layout).
	// Works on the device images: upload edited host flags first; the host mirror of flags is refreshed afterwards, like the reference does (FX/lbm.cpp:562).
	void voxelize_triangles_on_device(const float* p0, const float* p1, const float* p2, const uint triangle_number, const float3& pmin, const float3& pmax, const uchar flag=TYPE_S, const uint direction=2u) {
		float bbu[16] = {0.0f};
		memcpy(&bbu[0], &triangle_number, sizeof(uint));
		bbu[1] = pmin.x-2.0f; bbu[2] = pmin.y-2.0f; bbu[3] = pmin.z-2.0f; bbu[4] = pmax.x+2.0f; bbu[5] = pmax.y+2.0f; bbu[6] = pmax.z+2.0f;
		const bool dump = luw_dump_enabled();
		if(dump) luw_dump_voxelize_call(handle, (ulong)Nx*Ny*Nz, direction, flag, p0, p1, p2, triangle_number, bbu); // test hook (LUW_DUMP_DIR): the call's inputs, for the oracle voxeliser
		luw_check(luw_voxelize_mesh(handle, direction, flag, p0, p1, p2, triangle_number, bbu));
		flags.read_from_device();
		if(dump) luw_dump_array("vox_flags_after", flags.data(), (ulong)Nx*Ny*Nz);
	}
#ifdef LUW_USE_REFERENCE_UTILITIES
	void voxelize_mesh_on_device(const Mesh* mesh, const uchar flag=TYPE_S) { voxelize_triangles_on_device((const float*)mesh->p0, (const float*)mesh->p1, (const float*)mesh->p2, mesh->triangle_number, mesh->pmin, mesh->pmax, flag); }
#endif
	bool uses_tiles() const { int t = 0; luw_check(luw_domain_step_kernel(handle, &t)); return t!=0; } // does stream_collide run the TMA-tiled kernel on this domain?
	luw_domain* get_handle() const { return handle; } // reference: get_device() hands out the OpenCL Device; here the C-ABI handle
	int get_device_ordinal() const { return device; }
#ifdef LUW_USE_REFERENCE_UTILITIES
	const Device& get_device() const { // FX/lbm.hpp:141; callers read .info (FX/info.cpp:233-241, FX/setup.cpp:4415-4424) or pass it on to Memory / Kernel (FX/setup.cpp:1034)
		luw_device_info di;
		luw_check(luw_get_device_info(device, &di));
		device_view.dom = handle;
		device_view.info.id = (uint)device; device_view.info.name = di.name; device_view.info.memory = (uint)(di.memory_bytes/1048576ull); device_view.info.memory_used = (uint)(device_memory_used()/1048576ull);
		device_view.info.compute_units = di.compute_units; device_view.info.clock_frequency = di.clock_mhz;
		return device_view;
	}
private:
	mutable Device device_view;
public:
#endif
	ulong device_memory_used() const { uint64_t b = 0ull; luw_domain_bytes(handle, &b); return (ulong)b; } // Device_Info::memory_used (FX/info.cpp:233-241)
	static uint lbm_features();
};

// ---------------------------------------------------------------------------------------------------------------- LBM (FX/lbm.hpp:223-633)
class LBM {
private:
	uint Nx=1u, Ny=1u, Nz=1u, Dx=1u, Dy=1u, Dz=1u;
	bool initialized = false;
	ulong pending_steps = 0ull; // reference-tree mode: steps enqueued since the last synchronisation (run() synchronises every LUW_SYNC_EVERY steps, not every step)
	std::chrono::time_point<std::chrono::high_resolution_clock> pending_t0;
	void dump_state(const char* tag); // test hook, see luw_dump_enabled
	void flush_pending(); // synchronise and credit the elapsed time to the pending steps (info.update once per step, like FX/lbm.cpp:1292-1312)
	std::vector<luw_domain*> handles;
	void construct(const uint Nx, const uint Ny, const uint Nz, const uint Dx, const uint Dy, const uint Dz, const float nu, const float fx, const float fy, const float fz, const float alpha, const float beta);
	void initialize(); // FX/lbm.cpp:1221-1260
	void do_time_step(); // FX/lbm.cpp:1262-1290
	void communicate(const int payload);
public:
	template<typename T> class Memory_Container { // FX/lbm.hpp:252-423: holds no data, stitches the domains' host mirrors into one global array
	private:
		ulong N = 0ull; uint d = 1u;
		LBM* lbm = nullptr;
		Memory<T>** buffers = nullptr;
		std::string name = ""; // "rho" / "u" / "flags": file names and SI conversion of the VTK writer (FX/lbm.hpp:254)
		uint Nx=1u, Ny=1u, Nz=1u, Dx=1u, Dy=1u, Dz=1u, D=1u, NxDx=1u, NyDy=1u, NzDz=1u, Hx=0u, Hy=0u, Hz=0u;
		ulong NxNy=1ull, local_Nx=1ull, local_Ny=1ull, local_Nz=1ull, local_N=1ull;
		T& reference(const ulong i, const uint dimension) { // FX/lbm.hpp:274-297: global index -> (domain, local index with halo offsets)
			if(D==1u) return buffers[0]->data()[i<N ? i+(ulong)dimension*N : i%N+(ulong)std::max((ulong)dimension, i/N)*N]; // same element; the common case (i < N) without the two 64-bit divisions -- the case driver calls this a few times per cell of the lattice
			const ulong global_i = i%N, tt = global_i%NxNy;
			const uint x = (uint)(tt%(ulong)Nx), y = (uint)(tt/(ulong)Nx), z = (uint)(global_i/NxNy);
			const uint px = x%NxDx, py = y%NyDy, pz = z%NzDz, dx = x/NxDx, dy = y/NyDy, dz = z/NzDz, domain = dx+(dy+dz*Dy)*Dx;
			const ulong local_i = (ulong)(px+Hx)+((ulong)(py+Hy)+(ulong)(pz+Hz)*local_Ny)*local_Nx;
			return buffers[domain]->data()[local_i+std::max(i/N, (ulong)dimension)*local_N];
		}
	public:
		class Pointer {
			Memory_Container* memory = nullptr; uint dimension = 0u;
		public:
			Pointer() {}
			Pointer(Memory_Container* memory, const uint dimension) : memory(memory), dimension(dimension) {}
			T& operator[](const ulong i) { return memory->reference(i, dimension); }
			const T& operator[](const ulong i) const { return memory->reference(i, dimension); }
		};
		Pointer x, y, z;
		Memory_Container() {}
		Memory_Container(LBM* lbm, Memory<T>** buffers, const std::string& name="") { bind(lbm, buffers, name); }
		void bind(LBM* lbm_, Memory<T>** buffers_, const std::string& name_="") {
			lbm = lbm_; buffers = buffers_; name = name_;
			N = lbm->get_N(); d = buffers[0]->dimensions();
			Nx = lbm->get_Nx(); Ny = lbm->get_Ny(); Nz = lbm->get_Nz(); Dx = lbm->get_Dx(); Dy = lbm->get_Dy(); Dz = lbm->get_Dz(); D = Dx*Dy*Dz;
			NxNy = (ulong)Nx*(ulong)Ny; NxDx = Nx/Dx; NyDy = Ny/Dy; NzDz = Nz/Dz; Hx = Dx>1u; Hy = Dy>1u; Hz = Dz>1u;
			local_Nx = (ulong)(NxDx+2u*Hx); local_Ny = (ulong)(NyDy+2u*Hy); local_Nz = (ulong)(NzDz+2u*Hz); local_N = local_Nx*local_Ny*local_Nz;
			x = Pointer(this, 0u); if(d>1u) y = Pointer(this, 1u); if(d>2u) z = Pointer(this, 2u);
		}
		void reset(const T value=(T)0) { for(uint i=0u; i<D; i++) buffers[i]->reset(value); }
		ulong length() const { return N; }
		uint dimensions() const { return d; }
		ulong range() const { return N*(ulong)d; }
		ulong capacity() const { return N*(ulong)d*sizeof(T); }
		T& operator[](const ulong i) { return reference(i, 0u); }
		const T& operator[](const ulong i) const { return const_cast<Memory_Container*>(this)->reference(i, 0u); }
		T operator()(const ulong i) const { return const_cast<Memory_Container*>(this)->reference(i, 0u); }
		T operator()(const ulong i, const uint dimension) const { return const_cast<Memory_Container*>(this)->reference(i, dimension); }
		void read_from_device() { // FX/lbm.hpp:406-412
			for(uint i=0u; i<D; i++) lbm->lbm_domain[i]->enqueue_update_fields();
			for(uint i=0u; i<D; i++) buffers[i]->enqueue_read_from_device();
			for(uint i=0u; i<D; i++) buffers[i]->finish_queue();
		}
		void write_to_device() { // FX/lbm.hpp:413-416
			for(uint i=0u; i<D; i++) buffers[i]->enqueue_write_to_device();
			for(uint i=0u; i<D; i++) buffers[i]->finish_queue();
		}
#ifdef LUW_USE_REFERENCE_UTILITIES
		// Binary legacy-VTK export, byte-compatible with FX/lbm.hpp:307-356,417-423 (tools_core reads these files): STRUCTURED_POINTS header, then the field
		// as big-endian array-of-structures in SI units, the lowest Nz_write layers only if asked for.
		void write_host_to_vtk(const string& path="", const bool convert_to_si_units=true, const bool print_saved_message=true, const uint Nz_write=0u) {
			const string filename = create_file_extension(default_filename(path, name, ".vtk", lbm->get_t()), ".vtk");
			float spacing = 1.0f; T factor = (T)1;
			if(convert_to_si_units) {
				spacing = units.si_x(1.0f);
				if(name=="rho") factor = (T)units.si_rho(1.0f);
				if(name=="u") factor = (T)units.si_u(1.0f);
			}
			const uint Nz_out = (Nz_write>0u&&Nz_write<Nz) ? Nz_write : Nz;
			const ulong points = (ulong)Nx*(ulong)Ny*(ulong)Nz_out;
			float3 origin = spacing*float3(0.5f-0.5f*(float)Nx, 0.5f-0.5f*(float)Ny, 0.5f-0.5f*(float)Nz);
			if(convert_to_si_units) origin += vtk_origin_shift;
			const string type = sizeof(T)==1u ? "unsigned_char" : "float"; // the two element types of this build's fields (flags; rho, u)
			const string header = "# vtk DataFile Version 3.0\nFluidX3D "+filename.substr(filename.rfind('/')+1)+"\nBINARY\nDATASET STRUCTURED_POINTS\n"
				"DIMENSIONS "+to_string(Nx)+" "+to_string(Ny)+" "+to_string(Nz_out)+"\nORIGIN "+to_string(origin.x)+" "+to_string(origin.y)+" "+to_string(origin.z)+"\n"
				"SPACING "+to_string(spacing)+" "+to_string(spacing)+" "+to_string(spacing)+"\nPOINT_DATA "+to_string(points)+"\nSCALARS data "+type+" "+to_string(d)+"\nLOOKUP_TABLE default\n";
			create_folder(filename);
			std::ofstream file(filename, std::ios::out|std::ios::binary);
			file.write(header.c_str(), (std::streamsize)header.length());
			const ulong chunk = 4194304ull; // points per write
			std::vector<T> data(chunk*(ulong)d);
			const bool kelvin = convert_to_si_units&&name=="T"; // temperature is an affine map, not a factor: units.si_T(T) = T*unit_K + offset (FX/lbm.hpp:343)
			for(ulong p0=0ull; p0<points; p0+=chunk) {
				const ulong np = points-p0<chunk ? points-p0 : chunk;
				parallel_for(np, [&](ulong i) { for(uint c=0u; c<d; c++) { const T v = reference(p0+i, c); data[i*(ulong)d+(ulong)c] = reverse_bytes(kelvin ? (T)units.si_T((float)v) : (T)(factor*v)); } });
				file.write((const char*)data.data(), (std::streamsize)(np*(ulong)d*sizeof(T)));
			}
			file.close();
			if(print_saved_message) { info.allow_printing.lock(); print_info("File \""+filename+"\" saved."); info.allow_printing.unlock(); }
		}
		void write_device_to_vtk(const string& path="", const bool convert_to_si_units=true, const bool print_saved_message=true, const uint Nz_write=0u) {
			read_from_device();
			write_host_to_vtk(path, convert_to_si_units, print_saved_message, Nz_write);
		}
#endif
	};

	LBM_Domain** lbm_domain = nullptr; // one LBM domain per GPU
	Memory_Container<float> rho, u;
	Memory_Container<uchar> flags;
	Memory_Container<float> T; // bound only with LUW_TEMPERATURE (FX/lbm.hpp:441, FX/lbm.cpp:1102)

	LBM(const uint Nx, const uint Ny, const uint Nz, const uint Dx, const uint Dy, const uint Dz, const float nu, const float fx=0.0f, const float fy=0.0f, const float fz=0.0f, const float sigma=0.0f, const float alpha=0.0f, const float beta=0.0f);
	LBM(const uint Nx, const uint Ny, const uint Nz, const float nu, const float fx=0.0f, const float fy=0.0f, const float fz=0.0f, const float sigma=0.0f, const float alpha=0.0f, const float beta=0.0f);
	LBM(const uint3 N, const uint Dx, const uint Dy, const uint Dz, const float nu, const float fx=0.0f, const float fy=0.0f, const float fz=0.0f, const float sigma=0.0f, const float alpha=0.0f, const float beta=0.0f);
	LBM(const uint3 N, const float nu, const float fx=0.0f, const float fy=0.0f, const float fz=0.0f, const float sigma=0.0f, const float alpha=0.0f, const float beta=0.0f);
	~LBM();
	LBM(const LBM&) = delete;
	LBM& operator=(const LBM&) = delete;

	void run(const ulong steps=max_ulong, const ulong total_steps=max_ulong); // FX/lbm.cpp:1292-1312; run(0) = initialise only
	void update_fields(); // FX/lbm.cpp:1314-1317
	void reset(); // FX/lbm.cpp:1319-1321

	uint get_Nx() const { return Nx; } uint get_Ny() const { return Ny; } uint get_Nz() const { return Nz; }
	ulong get_N() const { return (ulong)Nx*(ulong)Ny*(ulong)Nz; }
	uint get_Dx() const { return Dx; } uint get_Dy() const { return Dy; } uint get_Dz() const { return Dz; }
	uint get_D() const { return Dx*Dy*Dz; }
	float get_nu() const { return lbm_domain[0]->get_nu(); }
	float get_tau() const { return 3.0f*get_nu()+0.5f; }
	float get_alpha() const { return lbm_domain[0]->get_alpha(); } float get_beta() const { return lbm_domain[0]->get_beta(); } float get_T_avg() const { return lbm_domain[0]->get_T_avg(); } // FX/lbm.hpp:483-485
	float get_fx() const { return lbm_domain[0]->get_fx(); } float get_fy() const { return lbm_domain[0]->get_fy(); } float get_fz() const { return lbm_domain[0]->get_fz(); }
	ulong get_t() const { return lbm_domain[0]->get_t(); }
	float get_Re_max() const { return 0.57735027f*sqrtf((float)Nx*(float)Nx+(float)Ny*(float)Ny+(float)Nz*(float)Nz)/get_nu(); } // Re < c*L_max/nu, FX/lbm.hpp:480
	float get_omega_x() const { return lbm_domain[0]->get_omega_x(); } float get_omega_y() const { return lbm_domain[0]->get_omega_y(); } float get_omega_z() const { return lbm_domain[0]->get_omega_z(); }
	uint get_velocity_set() const { return 19u; }
	void set_fx(const float fx) { for(uint d=0u; d<get_D(); d++) lbm_domain[d]->set_fx(fx); }
	void set_fy(const float fy) { for(uint d=0u; d<get_D(); d++) lbm_domain[d]->set_fy(fy); }
	void set_fz(const float fz) { for(uint d=0u; d<get_D(); d++) lbm_domain[d]->set_fz(fz); }
	void set_f(const float fx, const float fy, const float fz) { for(uint d=0u; d<get_D(); d++) lbm_domain[d]->set_f(fx, fy, fz); }
	void set_coriolis(const float omega_x, const float omega_y, const float omega_z) { for(uint d=0u; d<get_D(); d++) lbm_domain[d]->set_coriolis(omega_x, omega_y, omega_z); } // FX/lbm.hpp:496-498

	void coordinates(const ulong n, uint& x, uint& y, uint& z) const { const ulong t = n%((ulong)Nx*(ulong)Ny); x = (uint)(t%(ulong)Nx); y = (uint)(t/(ulong)Nx); z = (uint)(n/((ulong)Nx*(ulong)Ny)); } // FX/lbm.hpp:500-505
	ulong index(const uint x, const uint y, const uint z) const { return (ulong)x+((ulong)y+(ulong)z*(ulong)Ny)*(ulong)Nx; }
#ifdef LUW_USE_REFERENCE_UTILITIES
	float3 mirror_position(const float3& p) const { // FX/lbm.hpp:531-537
		return float3(sign(p.x)*(fmod(fabs(p.x)+0.5f*(float)Nx, (float)Nx)-0.5f*(float)Nx), sign(p.y)*(fmod(fabs(p.y)+0.5f*(float)Ny, (float)Ny)-0.5f*(float)Ny), sign(p.z)*(fmod(fabs(p.z)+0.5f*(float)Nz, (float)Nz)-0.5f*(float)Nz));
	}
	void coordinates(const float3& p, uint& x, uint& y, uint& z) const { // closest grid point of a position, FX/lbm.hpp:506-511
		const float3 mp = mirror_position(p);
		x = (uint)(mp.x+1.5f*(float)Nx)%Nx; y = (uint)(mp.y+1.5f*(float)Ny)%Ny; z = (uint)(mp.z+1.5f*(float)Nz)%Nz;
	}
	ulong index(const uint3 xyz) const { return index(xyz.x, xyz.y, xyz.z); }
	// LBM::voxelize_mesh_on_device, FX/lbm.cpp:1411-1645, for resting geometry, TYPE_S along z: with several domains every domain casts its rays against ITS subset of
	// the triangles (voxelize_triangles_on_device below: the reference's culling, including its skip of domains with an empty subset) inside the whole mesh's bounding
	// box; then the host mirrors are refreshed like FX/lbm.cpp:1641-1644 does before initialisation.
	void voxelize_mesh_on_device(const Mesh* mesh, const uchar flag=TYPE_S, const float3& rotation_center=float3(0.0f), const float3& linear_velocity=float3(0.0f), const float3& rotational_velocity=float3(0.0f)) {
		(void)rotation_center;
		if(length(linear_velocity)>0.0f||length(rotational_velocity)>0.0f) print_error("voxelize_mesh_on_device: moving geometry is not part of this build (LUW voxelises resting meshes only).");
		const std::vector<uint> subset = voxelize_triangles_on_device((const float*)mesh->p0, (const float*)mesh->p1, (const float*)mesh->p2, mesh->triangle_number, mesh->pmin, mesh->pmax, flag);
		if(get_D()>1u) { // FX/lbm.cpp:1604-1619
			ulong sum = 0ull; uint lo = subset[0], hi = subset[0];
			for(const uint n : subset) { sum += (ulong)n; lo = min(lo, n); hi = max(hi, n); }
			print_info("Voxelize pass 2 triangle subsets: min="+to_string(lo)+", max="+to_string(hi)+", sum="+to_string(sum)+", d0="+to_string(subset[0])+", est peak MB/GPU="+to_string((float)hi*36.0f/1048576.0f, 2u));
		}
		if(!initialized) { flags.read_from_device(); u.read_from_device(); }
		if(flag==TYPE_S) { // FX/lbm.cpp:1626-1637
			ulong solid = 0ull;
			const ulong N = get_N();
			for(ulong n=0ull; n<N; n++) if(flags[n]&TYPE_S) solid++;
			print_info("Voxelized cells (whole domain global, no halos): solid = "+to_string(solid)+", fluid = "+to_string(N-solid)+", total = "+to_string(N)+".");
		}
	}
	struct { int visualization_modes = 0; } graphics; // FX/setup.cpp:4125 sets it unconditionally; rendering is not part of this build
#endif
	// The stand-alone form of the above: triangles as 3 floats each, bounding box of the WHOLE mesh (the kernel's ray range, FX/lbm.cpp:497). Returns the number of
	// triangles each domain was given (the whole mesh for a single domain, FX/lbm.cpp:1488-1491).
	std::vector<uint> voxelize_triangles_on_device(const float* p0, const float* p1, const float* p2, const uint triangle_number, const float3& pmin, const float3& pmax, const uchar flag=TYPE_S, const uint direction=2u) {
		std::vector<uint> given(get_D(), triangle_number);
		if(get_D()==1u) { lbm_domain[0]->voxelize_triangles_on_device(p0, p1, p2, triangle_number, pmin, pmax, flag, direction); return given; }
		for(uint d=0u; d<get_D(); d++) {
			LBM_Domain* dom = lbm_domain[d];
			const std::vector<uint> ids = luw_cull_triangles(p0, p1, p2, triangle_number, direction, dom->get_Ox(), dom->get_Oy(), dom->get_Oz(), dom->get_Nx(), dom->get_Ny(), dom->get_Nz());
			given[d] = (uint)ids.size();
			if(ids.empty()) continue; // FX/lbm.cpp:499: no pass at all for this domain
			if(ids.size()==(size_t)triangle_number) { dom->voxelize_triangles_on_device(p0, p1, p2, triangle_number, pmin, pmax, flag, direction); continue; } // FX/lbm.cpp:1583
			std::vector<float> q0(3u*ids.size()), q1(3u*ids.size()), q2(3u*ids.size()); // subset in mesh order, FX/lbm.cpp:510-522
			for(size_t i=0u; i<ids.size(); i++) for(uint k=0u; k<3u; k++) { q0[3u*i+k] = p0[3u*ids[i]+k]; q1[3u*i+k] = p1[3u*ids[i]+k]; q2[3u*i+k] = p2[3u*ids[i]+k]; }
			dom->voxelize_triangles_on_device(q0.data(), q1.data(), q2.data(), (uint)ids.size(), pmin, pmax, flag, direction);
		}
		return given;
	}
	float3 position(const uint x, const uint y, const uint z) const { return float3((float)x-0.5f*(float)Nx+0.5f, (float)y-0.5f*(float)Ny+0.5f, (float)z-0.5f*(float)Nz+0.5f); }
	float3 position(const ulong n) const { uint x, y, z; coordinates(n, x, y, z); return position(x, y, z); }
	float3 size() const { return float3((float)Nx, (float)Ny, (float)Nz); }
	float3 center() const { return float3(0.5f*(float)Nx-0.5f, 0.5f*(float)Ny-0.5f, 0.5f*(float)Nz-0.5f); }
private:
	std::vector<Memory<float>*> rho_buffers, u_buffers, T_buffers;
	std::vector<Memory<uchar>*> flags_buffers;
};

// ---------------------------------------------------------------------------------------------------------------- running statistics (FX/setup.cpp:4441-4488)
// The averaging window of the case driver without its per-sample read-back: accumulate() updates mean / M2 of u and the mean of rho of every domain on the
// device (luw_stats_accumulate), download() returns them once, stitched over the global lattice in the reference's layout
// (avg_u interleaved [3n+c], avg_rho[n], M2_u / M2_v / M2_w[n]; FX/setup.cpp:4252-4266), ready for write_avg_vtk.
class LBM_Statistics {
private:
	LBM* lbm = nullptr;
	std::vector<luw_stats*> st;
public:
	explicit LBM_Statistics(LBM& lbm_) : lbm(&lbm_) {
		for(uint d=0u; d<lbm->get_D(); d++) { luw_stats* h = nullptr; luw_check(luw_stats_create(lbm->lbm_domain[d]->get_handle(), &h)); st.push_back(h); }
	}
	~LBM_Statistics() { for(luw_stats* h : st) luw_stats_destroy(h); }
	LBM_Statistics(const LBM_Statistics&) = delete;
	LBM_Statistics& operator=(const LBM_Statistics&) = delete;
	void accumulate() { // FX/setup.cpp:4411-4425 + 4441-4488: update_fields first when rho / u are not stored every step
		for(uint d=0u; d<lbm->get_D(); d++) lbm->lbm_domain[d]->enqueue_update_fields();
		for(uint d=0u; d<lbm->get_D(); d++) luw_check(luw_stats_accumulate(st[d]));
	}
	void reset() { for(luw_stats* h : st) luw_check(luw_stats_reset(h)); } // FX/setup.cpp:4556-4562
	ulong download(std::vector<float>& avg_u, std::vector<float>& avg_rho, std::vector<float>& M2_u, std::vector<float>& M2_v, std::vector<float>& M2_w) {
		const ulong N = lbm->get_N();
		avg_u.assign(3ull*N, 0.0f); avg_rho.assign(N, 0.0f); M2_u.assign(N, 0.0f); M2_v.assign(N, 0.0f); M2_w.assign(N, 0.0f);
		const uint Dx = lbm->get_Dx(), Dy = lbm->get_Dy(), Dz = lbm->get_Dz(), Hx = Dx>1u, Hy = Dy>1u, Hz = Dz>1u;
		uint64_t count = 0ull;
		for(uint d=0u; d<lbm->get_D(); d++) {
			const LBM_Domain* dom = lbm->lbm_domain[d];
			const ulong Nl = dom->get_N();
			std::vector<float> mu(3ull*Nl), m2(3ull*Nl), mr(Nl);
			luw_check(luw_stats_download(st[d], mu.data(), m2.data(), mr.data(), &count));
			for(uint z=Hz; z<dom->get_Nz()-Hz; z++) for(uint y=Hy; y<dom->get_Ny()-Hy; y++) for(uint x=Hx; x<dom->get_Nx()-Hx; x++) { // halo layers belong to the neighbours
				const ulong l = (ulong)x+((ulong)y+(ulong)z*(ulong)dom->get_Ny())*(ulong)dom->get_Nx();
				const ulong n = lbm->index((uint)((int)x+dom->get_Ox()), (uint)((int)y+dom->get_Oy()), (uint)((int)z+dom->get_Oz()));
				avg_u[3ull*n] = mu[l]; avg_u[3ull*n+1ull] = mu[Nl+l]; avg_u[3ull*n+2ull] = mu[2ull*Nl+l];
				M2_u[n] = m2[l]; M2_v[n] = m2[Nl+l]; M2_w[n] = m2[2ull*Nl+l];
				avg_rho[n] = mr[l];
			}
		}
		return (ulong)count;
	}
	void download_T(std::vector<float>& avg_T) { // the reference's avg_T (FX/setup.cpp:4262, 4481-4486), stitched like avg_rho; needs LUW_TEMPERATURE
		const ulong N = lbm->get_N();
		avg_T.assign(N, 0.0f);
		const uint Hx = lbm->get_Dx()>1u, Hy = lbm->get_Dy()>1u, Hz = lbm->get_Dz()>1u;
		for(uint d=0u; d<lbm->get_D(); d++) {
			const LBM_Domain* dom = lbm->lbm_domain[d];
			std::vector<float> mt(dom->get_N());
			luw_check(luw_stats_download_temperature(st[d], mt.data()));
			for(uint z=Hz; z<dom->get_Nz()-Hz; z++) for(uint y=Hy; y<dom->get_Ny()-Hy; y++) for(uint x=Hx; x<dom->get_Nx()-Hx; x++) {
				const ulong l = (ulong)x+((ulong)y+(ulong)z*(ulong)dom->get_Ny())*(ulong)dom->get_Nx();
				avg_T[lbm->index((uint)((int)x+dom->get_Ox()), (uint)((int)y+dom->get_Oy()), (uint)((int)z+dom->get_Oz()))] = mt[l];
			}
		}
	}
};

// [y*Nx + x] over the global columns: global z of the lowest non-solid cell over the blocks stacked in z (luw_column_ground per domain, minimum per column),
// 0xFFFFFFFF if none
inline std::vector<uint> luw_global_column_ground(LBM& lbm) {
	const uint Nx = lbm.get_Nx(), Ny = lbm.get_Ny(), Hx = lbm.get_Dx()>1u, Hy = lbm.get_Dy()>1u;
	std::vector<uint> ground((size_t)Nx*Ny, 0xFFFFFFFFu);
	for(uint d=0u; d<lbm.get_D(); d++) {
		const LBM_Domain* dom = lbm.lbm_domain[d];
		std::vector<uint32_t> g((size_t)dom->get_Nx()*dom->get_Ny());
		luw_check(luw_column_ground(dom->get_handle(), g.data()));
		for(uint y=Hy; y<dom->get_Ny()-Hy; y++) for(uint x=Hx; x<dom->get_Nx()-Hx; x++) {
			uint& G = ground[(size_t)(y+dom->get_Oy())*Nx+(size_t)(x+dom->get_Ox())];
			G = std::min(G, (uint)g[(size_t)y*dom->get_Nx()+x]);
		}
	}
	return ground;
}

// ---------------------------------------------------------------------------------------------------------------- pedestrian-level wind statistics (no reference counterpart)
// Surface-following layers: for every height h_k (cells) above the local ground or roof, the running mean and co-moments of u, mean / M2 / peak of the speed |u| and
// how many samples exceed each threshold (lattice units, at most LUW_WIND_MAX_THRESHOLDS), accumulated on the device per sample (luw_wind_stats_*). Construct it once the
// flags are on the device (after run(0)). The ground of a global column is the lowest non-solid cell over the domains stacked in z (luw_column_ground, minimum per
// column); each domain lists its owned plain-fluid cells ((flags & 0x03) == 0) at ground + h_k, read through a cell set, so no host mirror is materialised.
// download() stitches the lists into global layer-major arrays [k][y][x] (Nx*Ny*K per quantity; components / thresholds outermost); slots that are not listed
// (solid, TYPE_E, above the lattice) are NaN in the float fields, 0 in the counters and 0 in `valid`. File output (VTK, NetCDF) is the caller's business.
class LBM_WindStatistics {
private:
	LBM* lbm = nullptr;
	std::vector<uint> heights;
	uint thresholds = 0u;
	std::vector<luw_wind_stats*> st;
	std::vector<std::vector<ulong>> slots; // per domain: global slot of every listed cell
public:
	std::vector<uint> ground; // [y*Nx + x] over the global columns: global z of the lowest non-solid cell, 0xFFFFFFFF if none
	LBM_WindStatistics(LBM& lbm_, std::vector<uint> heights_in_cells, std::vector<float> thresholds_lattice) : lbm(&lbm_), heights(std::move(heights_in_cells)), thresholds((uint)thresholds_lattice.size()) {
		const uint Nx = lbm->get_Nx(), Ny = lbm->get_Ny(), Nz = lbm->get_Nz(), Hx = lbm->get_Dx()>1u, Hy = lbm->get_Dy()>1u, Hz = lbm->get_Dz()>1u;
		ground = luw_global_column_ground(*lbm);
		for(uint d=0u; d<lbm->get_D(); d++) {
			const LBM_Domain* dom = lbm->lbm_domain[d];
			const ulong lNx = dom->get_Nx(), lNy = dom->get_Ny();
			std::vector<uint64_t> cand; std::vector<ulong> cand_slot;
			for(size_t k=0u; k<heights.size(); k++) for(uint y=Hy; y<dom->get_Ny()-Hy; y++) for(uint x=Hx; x<dom->get_Nx()-Hx; x++) {
				const ulong gx = (ulong)(x+dom->get_Ox()), gy = (ulong)(y+dom->get_Oy());
				const uint G = ground[gy*Nx+gx];
				if(G==0xFFFFFFFFu||(ulong)G+heights[k]>=(ulong)Nz) continue;
				const long lz = (long)G+(long)heights[k]-(long)dom->get_Oz();
				if(lz<(long)Hz||lz>=(long)(dom->get_Nz()-Hz)) continue; // owned by another block
				cand.push_back((uint64_t)x+((uint64_t)y+(uint64_t)lz*lNy)*lNx);
				cand_slot.push_back((ulong)k*Nx*Ny+gy*Nx+gx);
			}
			std::vector<uint8_t> fl(cand.size());
			if(!cand.empty()) { // the candidates' flags, gathered on the device
				luw_cellset* cs = nullptr;
				luw_check(luw_cellset_create(dom->get_handle(), cand.size(), cand.data(), &cs));
				luw_check(luw_cellset_download(cs, LUW_FIELD_FLAGS, fl.data()));
				luw_check(luw_sync(dom->get_handle()));
				luw_check(luw_cellset_destroy(cs));
			}
			std::vector<uint64_t> cells; std::vector<ulong> sl;
			for(size_t i=0u; i<cand.size(); i++) if((fl[i]&0x03u)==0u) { cells.push_back(cand[i]); sl.push_back(cand_slot[i]); }
			luw_wind_stats* h = nullptr;
			luw_check(luw_wind_stats_create(dom->get_handle(), cells.size(), cells.data(), thresholds, thresholds_lattice.data(), &h));
			st.push_back(h); slots.push_back(std::move(sl));
		}
	}
	~LBM_WindStatistics() { for(luw_wind_stats* h : st) luw_wind_stats_destroy(h); }
	LBM_WindStatistics(const LBM_WindStatistics&) = delete;
	LBM_WindStatistics& operator=(const LBM_WindStatistics&) = delete;
	void accumulate() { // like LBM_Statistics::accumulate: update_fields first when rho / u are not stored every step
		for(uint d=0u; d<lbm->get_D(); d++) lbm->lbm_domain[d]->enqueue_update_fields();
		for(uint d=0u; d<lbm->get_D(); d++) luw_check(luw_wind_stats_accumulate(st[d]));
	}
	void reset() { for(luw_wind_stats* h : st) luw_check(luw_wind_stats_reset(h)); }
	// mean_u[c*M + m] (c = u v w), comoment[j*M + m] (j = uu vv ww uv uw vw), mean / M2 / max speed[m], exceed[j*M + m] (j < thresholds), valid[m]; m = k*Nx*Ny + y*Nx + x,
	// M = K*Nx*Ny. Returns the sample count.
	ulong download(std::vector<float>& mean_u, std::vector<float>& comoment, std::vector<float>& mean_speed, std::vector<float>& m2_speed, std::vector<float>& max_speed,
		std::vector<uint>& exceed, std::vector<uchar>& valid) {
		const ulong M = (ulong)heights.size()*lbm->get_Nx()*lbm->get_Ny();
		const float nan = std::nanf("");
		mean_u.assign(3ull*M, nan); comoment.assign(6ull*M, nan); mean_speed.assign(M, nan); m2_speed.assign(M, nan); max_speed.assign(M, nan);
		exceed.assign((ulong)thresholds*M, 0u); valid.assign(M, (uchar)0);
		uint64_t samples = 0ull;
		for(uint d=0u; d<lbm->get_D(); d++) {
			const std::vector<ulong>& sl = slots[d];
			const ulong K = sl.size();
			std::vector<float> mu(3ull*K), cm(6ull*K), ms(K), m2(K), mx(K);
			std::vector<uint32_t> ex((ulong)thresholds*K);
			luw_check(luw_wind_stats_download(st[d], mu.data(), cm.data(), ms.data(), m2.data(), mx.data(), ex.data(), &samples));
			for(ulong i=0ull; i<K; i++) {
				const ulong m = sl[i];
				for(ulong c=0ull; c<3ull; c++) mean_u[c*M+m] = mu[c*K+i];
				for(ulong j=0ull; j<6ull; j++) comoment[j*M+m] = cm[j*K+i];
				mean_speed[m] = ms[i]; m2_speed[m] = m2[i]; max_speed[m] = mx[i];
				for(ulong j=0ull; j<thresholds; j++) exceed[j*M+m] = ex[j*K+i];
				valid[m] = 1u;
			}
		}
		return (ulong)samples;
	}
};

// ---------------------------------------------------------------------------------------------------------------- wind loads on buildings (momentum exchange)
// Per sample and label (building): the force of the fluid on the label's surface cells and its moment about the label's reference point r0, [Fx Fy Fz Mx My Mz]
// in double, lattice units, GAUGE (relative to the reference pressure 1/3); per surface cell the running mean / M2 of the force (luw_solid_surface,
// luw_wall_loads_*; definitions in csrc/lbm_wall_loads.cuh). Construct it once the flags are on the device (after run(0)); call accumulate() after a step --
// no update_fields is needed. The same labels and r0 as lbm.WallLoads in Python: a building column is one whose global column ground (luw_global_column_ground)
// lies above ground_z + 1; building columns form 4-connected footprints (no wrap across the lattice edges) numbered 1..B in row-major (y, x) order of first
// appearance; a listed cell takes its column's label above z = ground_z, 0 (terrain) at or below it; r0 = the footprint's column-centre centroid at
// z = ground_z + 0.5 (overturning moment), the origin for label 0. column_labels[y*Nx + x] / ref_points[3*l + a] replace the defaults when not empty.
// The samples stay on the device until `capacity` are pending; then they are drained (the only host synchronisation). This class does not add the
// reference's FORCE_FIELD names (lbm.F, object_force, object_torque).
class LBM_WallLoads {
private:
	LBM* lbm = nullptr;
	uint capacity = 256u;
	ulong pending = 0ull;
	std::vector<luw_wall_loads*> st;
	std::vector<std::vector<ulong>> global; // per domain: global cell index of every listed cell, in list order
	std::vector<std::vector<uint>> labels_of; // per domain: label of every listed cell, in list order
	std::vector<double> loads; // drained samples [s][L][6], summed over the domains in domain order
	void drain() {
		const ulong S6 = (ulong)L*6ull;
		std::vector<double> total, part((ulong)capacity*S6);
		uint64_t n = 0ull;
		for(uint d=0u; d<st.size(); d++) {
			luw_check(luw_wall_loads_drain(st[d], part.data(), &n));
			if(d==0u) total.assign(part.begin(), part.begin()+(long)(n*S6));
			else for(ulong q=0ull; q<n*S6; q++) total[q] += part[q];
		}
		loads.insert(loads.end(), total.begin(), total.end());
		pending = 0ull;
	}
public:
	uint L = 0u; // labels
	std::vector<uint> ground; // [y*Nx + x]: global column ground
	std::vector<uint> column_labels; // [y*Nx + x]
	std::vector<double> ref_points; // [3*l + a]
	LBM_WallLoads(LBM& lbm_, const uint ground_z=0u, std::vector<uint> column_labels_in={}, std::vector<double> ref_points_in={}, const bool periodic_x=false,
		const bool periodic_y=false, const bool periodic_z=false, const uint capacity_=256u) : lbm(&lbm_), capacity(capacity_) {
		const uint Nx = lbm->get_Nx(), Ny = lbm->get_Ny();
		const uint periodic = (periodic_x ? 1u : 0u)|(periodic_y ? 2u : 0u)|(periodic_z ? 4u : 0u);
		ground = luw_global_column_ground(*lbm);
		if(column_labels_in.empty()) { // breadth-first flood fill, started in row-major order
			column_labels.assign((size_t)Nx*Ny, 0u);
			uint next = 0u;
			std::vector<ulong> queue;
			for(ulong s=0ull; s<(ulong)Nx*Ny; s++) {
				if(!((ulong)ground[s]>(ulong)ground_z+1ull)||column_labels[s]!=0u) continue;
				column_labels[s] = ++next;
				queue.assign(1u, s);
				for(size_t q=0u; q<queue.size(); q++) {
					const ulong c = queue[q], x = c%Nx, y = c/Nx;
					const ulong nb[4] = { y>0ull ? c-Nx : c, y+1ull<Ny ? c+Nx : c, x>0ull ? c-1ull : c, x+1ull<Nx ? c+1ull : c };
					for(const ulong m : nb) if(m!=c&&(ulong)ground[m]>(ulong)ground_z+1ull&&column_labels[m]==0u) { column_labels[m] = next; queue.push_back(m); }
				}
			}
		} else {
			column_labels = std::move(column_labels_in);
		}
		L = 1u;
		for(const uint l : column_labels) L = std::max(L, l+1u);
		if(ref_points_in.empty()) {
			std::vector<ulong> cnt(L, 0ull), sx(L, 0ull), sy(L, 0ull);
			for(ulong s=0ull; s<(ulong)Nx*Ny; s++) { const uint l = column_labels[s]; cnt[l]++; sx[l] += s%Nx; sy[l] += s/Nx; }
			ref_points.assign(3ull*L, 0.0);
			for(uint l=1u; l<L; l++) if(cnt[l]>0ull) {
				ref_points[3u*l] = (double)sx[l]/(double)cnt[l]; ref_points[3u*l+1u] = (double)sy[l]/(double)cnt[l]; ref_points[3u*l+2u] = (double)ground_z+0.5;
			}
		} else {
			ref_points = std::move(ref_points_in);
		}
		for(uint d=0u; d<lbm->get_D(); d++) {
			const LBM_Domain* dom = lbm->lbm_domain[d];
			const ulong lNx = dom->get_Nx(), lNy = dom->get_Ny();
			uint64_t count = 0ull;
			luw_check(luw_solid_surface(dom->get_handle(), periodic, 0ull, nullptr, &count));
			std::vector<uint64_t> cells(count);
			luw_check(luw_solid_surface(dom->get_handle(), periodic, count, cells.data(), &count));
			std::vector<uint> lab(count);
			std::vector<ulong> gidx(count), order(count);
			for(ulong k=0ull; k<count; k++) {
				const ulong n = cells[k];
				const ulong gx = (ulong)((long)(n%lNx)+dom->get_Ox()), gy = (ulong)((long)((n/lNx)%lNy)+dom->get_Oy()), gz = (ulong)((long)(n/(lNx*lNy))+dom->get_Oz());
				lab[k] = gz>(ulong)ground_z ? column_labels[gy*Nx+gx] : 0u;
				gidx[k] = gx+(gy+gz*Ny)*(ulong)Nx;
				order[k] = k;
			}
			std::sort(order.begin(), order.end(), [&](const ulong a, const ulong b) { return lab[a]!=lab[b] ? lab[a]<lab[b] : cells[a]<cells[b]; });
			std::vector<uint64_t> sc(count); std::vector<uint32_t> sl(count); std::vector<ulong> sg(count); std::vector<uint> slab(count);
			for(ulong k=0ull; k<count; k++) { sc[k] = cells[order[k]]; sl[k] = lab[order[k]]; sg[k] = gidx[order[k]]; slab[k] = lab[order[k]]; }
			luw_wall_loads* h = nullptr;
			luw_check(luw_wall_loads_create(dom->get_handle(), count, sc.data(), sl.data(), L, ref_points.data(), periodic, capacity, &h));
			st.push_back(h); global.push_back(std::move(sg)); labels_of.push_back(std::move(slab));
		}
	}
	~LBM_WallLoads() { for(luw_wall_loads* h : st) luw_wall_loads_destroy(h); }
	LBM_WallLoads(const LBM_WallLoads&) = delete;
	LBM_WallLoads& operator=(const LBM_WallLoads&) = delete;
	void accumulate() {
		if(pending==(ulong)capacity) drain();
		for(uint d=0u; d<lbm->get_D(); d++) luw_check(luw_wall_loads_accumulate(st[d], lbm->lbm_domain[d]->get_t()));
		pending++;
	}
	void reset() { for(luw_wall_loads* h : st) luw_check(luw_wall_loads_reset(h)); pending = 0ull; loads.clear(); }
	// series[(s*L + l)*6 + a], a = Fx Fy Fz Mx My Mz, since construction / reset. Returns the sample count.
	ulong series(std::vector<double>& out) {
		drain();
		out = loads;
		return (ulong)(loads.size()/((ulong)L*6ull));
	}
	// all listed cells in ascending global index n = x+(y+z*Ny)*Nx: cell[k], label[k], mean_F[a*K + k], m2_F[a*K + k]. Returns the sample count.
	ulong surface(std::vector<ulong>& cell, std::vector<uint>& label, std::vector<float>& mean_F, std::vector<float>& m2_F) {
		std::vector<ulong> all; std::vector<uint> lab; std::vector<float> mean[3], m2[3];
		uint64_t samples = 0ull;
		for(uint d=0u; d<st.size(); d++) {
			const ulong K = global[d].size();
			std::vector<float> a(3ull*K), b(3ull*K);
			luw_check(luw_wall_loads_download_cells(st[d], a.data(), b.data(), &samples));
			all.insert(all.end(), global[d].begin(), global[d].end()); lab.insert(lab.end(), labels_of[d].begin(), labels_of[d].end());
			for(uint c=0u; c<3u; c++) { mean[c].insert(mean[c].end(), a.begin()+(long)(c*K), a.begin()+(long)((c+1u)*K)); m2[c].insert(m2[c].end(), b.begin()+(long)(c*K), b.begin()+(long)((c+1u)*K)); }
		}
		const ulong K = all.size();
		std::vector<ulong> order(K);
		for(ulong k=0ull; k<K; k++) order[k] = k;
		std::sort(order.begin(), order.end(), [&](const ulong a, const ulong b) { return all[a]<all[b]; });
		cell.resize(K); label.resize(K); mean_F.resize(3ull*K); m2_F.resize(3ull*K);
		for(ulong k=0ull; k<K; k++) {
			cell[k] = all[order[k]]; label[k] = lab[order[k]];
			for(uint c=0u; c<3u; c++) { mean_F[c*K+k] = mean[c][order[k]]; m2_F[c*K+k] = m2[c][order[k]]; }
		}
		return (ulong)samples;
	}
};
