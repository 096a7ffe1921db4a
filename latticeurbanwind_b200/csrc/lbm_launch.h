// Host-side launch interface between the C ABI (luw_cabi.cu) and the two arithmetic builds of the kernels.
#pragma once
#include <cuda.h>
#include <type_traits>
#include <utility>
#include "lbm_common.cuh"

namespace luw {
struct ParticleSet; // lbm_particles.cuh
// Run-time value -> template argument: f is called with the matching value as a std::integral_constant (decltype(arg)::value names the instantiation).
// precision p; unknown values take FP16C
template<class F> auto with_precision(const int p, F&& f) {
	switch(p) {
		case P_FP32: return f(std::integral_constant<int, P_FP32>{});
		case P_FP16S: return f(std::integral_constant<int, P_FP16S>{});
		default: return f(std::integral_constant<int, P_FP16C>{});
	}
}
// the S of the list equal to x; cudaErrorInvalidValue when there is none
template<class T, T... S, class F> cudaError_t with_value(const T x, F&& f, std::integer_sequence<T, S...>) {
	cudaError_t e = cudaErrorInvalidValue;
	(void)((x==S&&(e = f(std::integral_constant<T, S>{}), true))||...);
	return e;
}
template<uint32_t... S, class F> cudaError_t with_feature_set(const uint32_t feat, F&& f) { return with_value(feat, f, std::integer_sequence<uint32_t, S...>{}); }

struct TileMaps { CUtensorMap fi, fiA, flags; }; // TMA descriptors: DDF array (4-D: x, y, z, slot) with one tile as box; the same with a box of nine slots at element stride 2; flag array (3-D)
struct TileShape { int tx, ty, tz; };
struct KernelSet { // one per arithmetic mode; every function enqueues exactly one kernel on `s` and returns the CUDA launch status
	cudaError_t (*initialize)(const DomainConst& c, cudaStream_t s);
	cudaError_t (*stream_collide)(const DomainConst& c, const StepArgs& a, cudaStream_t s);
	cudaError_t (*update_fields)(const DomainConst& c, const StepArgs& a, cudaStream_t s);
	cudaError_t (*halo_fi)(const DomainConst& c, int precision, uint32_t axis, uint32_t odd, bool insert, bool xfast, void* buf_p, void* buf_m, cudaStream_t s); // xfast: payload in thread order (library-internal buffers) instead of the reference's face order
	cudaError_t (*halo_rho_u_flags)(const DomainConst& c, uint32_t axis, bool insert, bool xfast, void* buf_p, void* buf_m, cudaStream_t s);
	cudaError_t (*vk_inlet_apply)(uint64_t Ncells, uint32_t use_interp, float t0, float t1, float alpha, uint64_t P, uint64_t M, uint64_t V,
		const uint64_t* point_cell, const uint8_t* point_face, const float* pd, const float* md, const float* cs, float* u, cudaStream_t s); // cs: A cos(phi), A sin(phi) table (FAST)
	// TMA-tiled stream_collide (lbm_tile.cuh): the tile variant a lattice of this precision, feature set and size runs -- `want` (< 0: the default) if it is
	// built for the feature set and its tile is not wider than the lattice, else the first fallback that is -- and its box shape; -1 if there is none
	int (*choose_tile)(int precision, uint32_t features, uint32_t Nx, uint32_t Ny, uint32_t Nz, int want, TileShape* shape);
	cudaError_t (*stream_collide_tile)(const DomainConst& c, const StepArgs& a, const TileMaps& maps, int variant, int sm_count, cudaStream_t s);
	cudaError_t (*voxelize)(const DomainConst& c, uint32_t direction, uint8_t flag, uint32_t ntri, const float* box6, const float* p0, const float* p1, const float* p2, cudaStream_t s); // p0..p2: device
	// the same through a bin grid over the face (csrc/vox_bins.h): bin_start[bins0*bins1 + 1], bin_ids[]: device
	cudaError_t (*voxelize_binned)(const DomainConst& c, uint32_t direction, uint8_t flag, uint32_t ntri, const float* box6, uint32_t bins0, uint32_t bins1, const uint32_t* bin_start, const uint32_t* bin_ids,
		const float* p0, const float* p1, const float* p2, cudaStream_t s);
	// thermal D3Q7 extension (domains created with LUW_TEMPERATURE): the three LBM kernels with the reference's TEMPERATURE blocks, halos of gi and T
	cudaError_t (*initialize_thermal)(const DomainConst& c, cudaStream_t s);
	cudaError_t (*stream_collide_thermal)(const DomainConst& c, const StepArgs& a, cudaStream_t s);
	cudaError_t (*update_fields_thermal)(const DomainConst& c, const StepArgs& a, cudaStream_t s);
	cudaError_t (*halo_gi)(const DomainConst& c, int precision, uint32_t axis, uint32_t odd, bool insert, bool xfast, void* buf_p, void* buf_m, cudaStream_t s);
	cudaError_t (*halo_T)(const DomainConst& c, uint32_t axis, bool insert, bool xfast, void* buf_p, void* buf_m, cudaStream_t s);
	cudaError_t (*thermal_g)(const DomainConst& c, const StepArgs& a, cudaStream_t s); // the TEMPERATURE block alone, after a tiled momentum step that filled c.upre
	// probe sample (lbm_probes.cuh): rho, u (and T) of `count` listed cells (device indices), as update_fields + a read would give them, into out[c*count + k]
	cudaError_t (*probe_sample)(const DomainConst& c, const StepArgs& a, uint64_t count, const uint64_t* cell, float* out, unsigned grid, cudaStream_t s);
	// tracer particles (lbm_particles.cuh): one advance of the ACTIVE particles of `s` by dt with the cell velocities probe_sample reads; call: the ring's advance count
	cudaError_t (*particles_advance)(const DomainConst& c, const StepArgs& a, const ParticleSet& s, uint64_t call, float dt, double sigma, unsigned grid, cudaStream_t st);
};
const KernelSet& kernels_strict(); // lbm_strict.cu: -fmad=false
const KernelSet& kernels_fast(); // lbm_fast.cu: contraction allowed
} // namespace luw
