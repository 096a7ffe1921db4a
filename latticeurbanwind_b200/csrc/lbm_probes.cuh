// Probe time series on the device: rho, u (and T) at a fixed list of cells, read from the DDFs of the current state without luw_update_fields over the lattice
// and without writing into it. A sample costs O(probes) instead of O(lattice); it leaves the domain's rho / u / T fields as they are.
//
// Per listed cell the kernel writes what luw_update_fields(t, ...) followed by a read of rho / u (/ T) at that cell gives:
//  * domains that store rho / u every step (UPDATE_FIELDS): the stored fields. (Inside nudging / sponge zones these are the step's values, which luw_force
//    forms with zones on; update_fields forms them with zones off.)
//  * cells update_fields skips (TYPE_S, TYPE_G) and the rho / u of TYPE_E cells under EQUILIBRIUM_BOUNDARIES: the stored fields;
//  * every other cell: update_fields_cell (lbm_kernels.cuh), the arithmetic update_fields itself runs, so that the value is the same bit for bit in the same
//    arithmetic build (this file is compiled into lbm_strict.cu and lbm_fast.cu through lbm_launch.inc).
// Output: one ring slot, out[c*count + k], c = rho, ux, uy, uz (and T on LUW_TEMPERATURE domains).
#pragma once
#include "lbm_kernels.cuh"

namespace luw {
namespace {

// FEAT: F_UPDATE_FIELDS alone, or a subset of F_VOLUME_FORCE | F_EQUILIBRIUM (the bits update_fields depends on). cell[k]: device (pitched) indices of owned cells.
template<int P, uint32_t FEAT, bool TH> __global__ void __launch_bounds__(256) k_probe_sample(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a,
	const uint64_t count, const uint64_t* __restrict__ cell, float* __restrict__ out) {
	constexpr bool UF = (FEAT&F_UPDATE_FIELDS)!=0u, EQ = (FEAT&F_EQUILIBRIUM)!=0u;
	for(uint64_t k=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; k<count; k+=(uint64_t)gridDim.x*blockDim.x) {
		const uint64_t n = cell[k];
		const uint32_t fl = c.flags[n], bo = fl&TYPE_BO;
		const bool computed = !UF&&bo!=TYPE_S&&(fl&TYPE_SU)!=TYPE_G;
		float rhon, uxn, uyn, uzn, Tn;
		if(computed) {
			const uint32_t x = (uint32_t)(n%c.Px), y = (uint32_t)((n/c.Px)%c.Ny), z = (uint32_t)(n/((uint64_t)c.Px*c.Ny));
			uint64_t j[Q];
			neighbors(c, x, y, z, j);
			update_fields_cell<P, FEAT, TH>(c, a, j, x, y, z, fl, rhon, uxn, uyn, uzn, Tn);
		}
		if(!computed||(EQ&&bo==TYPE_E)) { rhon = c.rho[n]; uxn = c.u[n]; uyn = c.u[c.N+n]; uzn = c.u[2ull*c.N+n]; }
		out[k] = rhon; out[count+k] = uxn; out[2ull*count+k] = uyn; out[3ull*count+k] = uzn;
		if constexpr(TH) out[4ull*count+k] = computed ? Tn : c.T[n]; // update_fields_thermal stores T of every executing cell (a TYPE_T cell's T is its preset)
	}
}

} // anonymous namespace
} // namespace luw
