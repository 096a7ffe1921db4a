// Pedestrian-level wind statistics on the device: per-sample accumulators restricted to a list of cells (typically a few layers at fixed heights above
// the local ground or roof). Extends the averaging window (luw_stats_*, the reference's FX/setup.cpp:4411-4542) with what users of an urban-wind LES evaluate
// at street and roof level and what cannot be rebuilt from mean / M2 per component: the full velocity co-moment matrix (u'w' and friends), the running mean,
// M2 and peak of the speed |u|, and threshold exceedance counts (comfort criteria). The reference has no counterpart; it would read the whole u field back
// per sample and loop on the host.
//
// Bit-exactness: every product and sum is rounded separately (__fmul_rn / __fadd_rn, __fsqrt_rn), so the kernel computes exactly what a float32 restatement
// without FMA computes (oracle/wind_stats_oracle.py), and its means and diagonal co-moments are those of k_stats_accumulate for the same cells.
#pragma once
#include <cstdint>

namespace luw {

constexpr uint32_t WIND_MAX_THRESHOLDS = 8u;
// float accumulators per listed cell, SoA [j*count + k]: mean u v w (0..2), co-moments uu vv ww uv uw vw (3..8), mean speed (9), M2 speed (10), max speed (11)
constexpr uint32_t WIND_FLOAT_ACCUMULATORS = 12u;
struct WindThresholds { float t[WIND_MAX_THRESHOLDS]; uint32_t count; }; // by value in the kernel parameters

// ground[y*Nx + x] = global z (Oz + z) of the lowest cell of local column (x, y) whose flags are not solid ((flags & 0x03) != TYPE_S) among the owned
// layers z0 <= z < z1 (the z halo layers of a decomposed axis belong to the neighbours), 0xFFFFFFFF if there is none. grid (ceil(Nx/256), Ny):
// threads of a warp take consecutive x, so every flag read of a warp is one coalesced row segment.
__global__ void __launch_bounds__(256) k_column_ground(const uint32_t Nx, const uint32_t Px, const uint32_t Ny, const uint32_t z0, const uint32_t z1, const int32_t Oz,
	const uint8_t* __restrict__ flags, uint32_t* __restrict__ ground) {
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y;
	if(x>=Nx) return;
	uint32_t g = 0xFFFFFFFFu;
	for(uint32_t z=z0; z<z1; z++) {
		if((flags[(uint64_t)x+((uint64_t)y+(uint64_t)z*Ny)*Px]&0x03u)!=0x01u) { g = (uint32_t)(Oz+(int32_t)z); break; }
	}
	ground[(uint64_t)y*Nx+x] = g;
}

// One sample: Welford update of the listed cells' accumulators with the running sample count n (inv_n = 1/n, rounded on the host like luw_stats_accumulate).
// u: the domain's pitched velocity field [c*N + n]; cell[k]: device index of listed cell k.
__global__ void __launch_bounds__(256) k_wind_stats_accumulate(const uint64_t count, const uint64_t N, const float inv_n, const float* __restrict__ u,
	const uint64_t* __restrict__ cell, const WindThresholds thr, float* __restrict__ acc, uint32_t* __restrict__ exceed) {
	for(uint64_t k=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; k<count; k+=(uint64_t)gridDim.x*blockDim.x) {
		const uint64_t n = cell[k];
		const float x[3] = { u[n], u[N+n], u[2ull*N+n] };
		float d[3], e[3];
#pragma unroll
		for(uint32_t c=0u; c<3u; c++) {
			float mean = acc[(uint64_t)c*count+k];
			d[c] = __fadd_rn(x[c], -mean); // old mean
			mean = __fadd_rn(mean, __fmul_rn(d[c], inv_n));
			e[c] = __fadd_rn(x[c], -mean); // new mean
			acc[(uint64_t)c*count+k] = mean;
		}
		const uint32_t a[6] = { 0u, 1u, 2u, 0u, 0u, 1u }, b[6] = { 0u, 1u, 2u, 1u, 2u, 2u }; // uu vv ww uv uw vw
#pragma unroll
		for(uint32_t j=0u; j<6u; j++) {
			float* p = acc+(uint64_t)(3u+j)*count+k;
			*p = __fadd_rn(*p, __fmul_rn(d[a[j]], e[b[j]]));
		}
		const float s = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(x[0], x[0]), __fmul_rn(x[1], x[1])), __fmul_rn(x[2], x[2])));
		float mean_s = acc[9ull*count+k];
		const float ds = __fadd_rn(s, -mean_s);
		mean_s = __fadd_rn(mean_s, __fmul_rn(ds, inv_n));
		acc[9ull*count+k] = mean_s;
		acc[10ull*count+k] = __fadd_rn(acc[10ull*count+k], __fmul_rn(ds, __fadd_rn(s, -mean_s)));
		acc[11ull*count+k] = fmaxf(acc[11ull*count+k], s);
#pragma unroll
		for(uint32_t j=0u; j<WIND_MAX_THRESHOLDS; j++) if(j<thr.count) exceed[(uint64_t)j*count+k] += s>thr.t[j] ? 1u : 0u;
	}
}

} // namespace luw
