// Wind loads on buildings, on the device: the momentum-exchange force of the fluid on every solid cell that touches the fluid, its moment about a reference
// point per label (building), a deterministic per-label sum per sample and per-cell surface statistics of the force. The reference's FORCE_FIELD extension
// (update_force_field + object_force / object_torque) stores a 12 B-per-cell force field over the whole lattice, reduces with float atomics (sums vary from
// run to run) and has no notion of "which building"; here only the listed surface cells are visited and every sum has a fixed order.
//
// Definitions (oracle/wall_loads_oracle.py restates them):
//  * counted link of DDF i at cell n: the cell the DDF streamed from, n - c_i, is not solid ((flags & 0x03) != TYPE_S), and reaching it does not cross a GLOBAL
//    lattice face of an axis the caller declares non-periodic (decided by global coordinates, so a decomposition boundary is never taken for the face);
//  * listed cell: an owned (non-halo) solid cell with at least one counted link;
//  * per-cell force F = 2 m, m the momentum sum of rho_u (lbm_common.cuh) over the DDFs load_f<P> reads at the solid cell with the time argument of the current
//    state (the one luw_update_fields is given), the term of a non-counted link replaced by +0.0 in place. The DDFs are stored shifted (f - w_i), so F is the
//    GAUGE load, relative to the reference pressure 1/3 (lattice units: rho = 1, one cell edge, one step);
//  * per-cell moment M = (r - r0) x F in double, r the cell's global integer coordinates, r0 the reference point of its label; every product and sum rounded
//    separately (__dmul_rn / __dadd_rn / __dsub_rn);
//  * label load per sample: sum of (F, M) over the label's cells in double, in a fixed order that depends on the list only: a thread sums a chunk of
//    WALL_CHUNK consecutive cells of one label in index order, a thread sums a group of up to WALL_GROUP consecutive chunks of one label in order, and one
//    thread per label and component sums the label's groups in order (three levels, so that the terrain label -- a million cells on a city lattice -- is not
//    one long serial chain). No atomics, no shuffles, no shared memory, so the same source runs on host threads (tests/host_emulation) with the same result.
#pragma once
#include <cstdint>
#include "lbm_kernels.cuh"

namespace luw {

constexpr uint32_t WALL_CHUNK = 32u; // listed cells per first-level partial sum
constexpr uint32_t WALL_GROUP = 32u; // first-level sums per second-level sum
constexpr uint32_t WALL_COMPONENTS = 6u; // Fx Fy Fz Mx My Mz per label and sample

// c_i of the D3Q19 DDF i in the order of neighbors() (lbm_common.cuh: j[i] = n + c_i)
__host__ __device__ __forceinline__ void wall_dir(const uint32_t i, int& cx, int& cy, int& cz) {
	const int X[19] = { 0, 1,-1, 0, 0, 0, 0, 1,-1, 1,-1, 0, 0, 1,-1, 1,-1, 0, 0 };
	const int Y[19] = { 0, 0, 0, 1,-1, 0, 0, 1,-1, 0, 0, 1,-1,-1, 1, 0, 0, 1,-1 };
	const int Z[19] = { 0, 0, 0, 0, 0, 1,-1, 0, 0, 1,-1, 1,-1, 0, 0,-1, 1,-1, 1 };
	cx = X[i]; cy = Y[i]; cz = Z[i];
}

// bit i (1 <= i < 19) set: the link of DDF i at the local cell (x, y, z) counts. periodic: bit a set = axis a is periodic.
__device__ __forceinline__ uint32_t wall_links(const DomainConst& c, const uint32_t periodic, const uint32_t x, const uint32_t y, const uint32_t z) {
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const int gx = (int)x+c.Ox, gy = (int)y+c.Oy, gz = (int)z+c.Oz;
	uint32_t m = 0u;
#pragma unroll
	for(uint32_t i=1u; i<(uint32_t)Q; i++) {
		int cx, cy, cz;
		wall_dir(i, cx, cy, cz);
		const uint32_t o = (i&1u) ? i+1u : i-1u; // j[o] = n - c_i
		const bool inside = ((periodic&1u)||(uint32_t)(gx-cx)<c.Nxg)&&((periodic&2u)||(uint32_t)(gy-cy)<c.Nyg)&&((periodic&4u)||(uint32_t)(gz-cz)<c.Nzg);
		if(inside&&(c.flags[j[o]]&0x03u)!=TYPE_S) m |= 1u<<i;
	}
	return m;
}

// Surface enumeration over the owned rows (y, z) (y0 <= y < y1, z0 <= z < z1, owned x0 <= x < x1), one thread per row scanning x upwards:
// offset == nullptr: count[r] = listed cells of row r = (y-y0) + (z-z0)*(y1-y0); otherwise the listed cells' local DENSE indices x+(y+z*Ny)*Nx are written
// from cells[offset[r]] on, in ascending order (rows are in ascending index order, so the whole list ascends).
__global__ void __launch_bounds__(256) k_surface_rows(const __grid_constant__ DomainConst c, const uint32_t periodic, const uint32_t x0, const uint32_t x1,
	const uint32_t y0, const uint32_t y1, const uint32_t z0, const uint32_t z1, const uint64_t* __restrict__ offset, uint32_t* __restrict__ count, uint64_t* __restrict__ cells) {
	const uint64_t rows = (uint64_t)(y1-y0)*(z1-z0);
	for(uint64_t r=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; r<rows; r+=(uint64_t)gridDim.x*blockDim.x) {
		const uint32_t y = y0+(uint32_t)(r%(y1-y0)), z = z0+(uint32_t)(r/(y1-y0));
		const uint8_t* row = c.flags+((uint64_t)y+(uint64_t)z*c.Ny)*c.Px;
		uint64_t k = offset ? offset[r] : 0ull;
		uint32_t n = 0u;
		for(uint32_t x=x0; x<x1; x++) {
			if((row[x]&0x03u)!=TYPE_S||wall_links(c, periodic, x, y, z)==0u) continue;
			if(offset) cells[k++] = (uint64_t)x+((uint64_t)y+(uint64_t)z*c.Ny)*c.Nx;
			n++;
		}
		if(!offset) count[r] = n;
	}
}

// links[k] of the listed cells (device indices cell[k]), classified once when the list is set up.
__global__ void __launch_bounds__(256) k_wall_links(const __grid_constant__ DomainConst c, const uint32_t periodic, const uint64_t count, const uint64_t* __restrict__ cell,
	uint32_t* __restrict__ links) {
	for(uint64_t k=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; k<count; k+=(uint64_t)gridDim.x*blockDim.x) {
		const uint64_t n = cell[k];
		const uint32_t x = (uint32_t)(n%c.Px), y = (uint32_t)((n/c.Px)%c.Ny), z = (uint32_t)(n/((uint64_t)c.Px*c.Ny));
		links[k] = wall_links(c, periodic, x, y, z);
	}
}

// One sample, per listed cell: F = 2 m (SoA F[a*count + k], a = x y z) and the Welford update of its mean / M2 (acc[a*count + k] mean, acc[(3+a)*count + k] M2)
// with the running sample count n (inv_n = 1/n, rounded on the host like luw_stats_accumulate). odd = t & 1 of the current state.
template<int P> __global__ void __launch_bounds__(256) k_wall_cells(const __grid_constant__ DomainConst c, const uint64_t count, const uint64_t* __restrict__ cell,
	const uint32_t* __restrict__ links, const uint32_t odd, const float inv_n, float* __restrict__ F, float* __restrict__ acc) {
	typedef typename Ddf<P>::T T;
	for(uint64_t k=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; k<count; k+=(uint64_t)gridDim.x*blockDim.x) {
		const uint64_t n = cell[k];
		const uint32_t x = (uint32_t)(n%c.Px), y = (uint32_t)((n/c.Px)%c.Ny), z = (uint32_t)(n/((uint64_t)c.Px*c.Ny));
		uint64_t j[Q];
		neighbors(c, x, y, z, j);
		float f[Q];
		load_f<P>((const T*)c.fi, c.N, j, odd, f);
		const uint32_t m = links[k];
#pragma unroll
		for(uint32_t i=0u; i<(uint32_t)Q; i++) if(!((m>>i)&1u)) f[i] = 0.0f;
		// the momentum sums of rho_u, left to right
		float mx = f[1];
		mx = __fsub_rn(mx, f[2]); mx = __fadd_rn(mx, f[7]); mx = __fsub_rn(mx, f[8]); mx = __fadd_rn(mx, f[9]); mx = __fsub_rn(mx, f[10]);
		mx = __fadd_rn(mx, f[13]); mx = __fsub_rn(mx, f[14]); mx = __fadd_rn(mx, f[15]); mx = __fsub_rn(mx, f[16]);
		float my = f[3];
		my = __fsub_rn(my, f[4]); my = __fadd_rn(my, f[7]); my = __fsub_rn(my, f[8]); my = __fadd_rn(my, f[11]); my = __fsub_rn(my, f[12]);
		my = __fadd_rn(my, f[14]); my = __fsub_rn(my, f[13]); my = __fadd_rn(my, f[17]); my = __fsub_rn(my, f[18]);
		float mz = f[5];
		mz = __fsub_rn(mz, f[6]); mz = __fadd_rn(mz, f[9]); mz = __fsub_rn(mz, f[10]); mz = __fadd_rn(mz, f[11]); mz = __fsub_rn(mz, f[12]);
		mz = __fadd_rn(mz, f[16]); mz = __fsub_rn(mz, f[15]); mz = __fadd_rn(mz, f[18]); mz = __fsub_rn(mz, f[17]);
		const float v[3] = { __fmul_rn(2.0f, mx), __fmul_rn(2.0f, my), __fmul_rn(2.0f, mz) };
#pragma unroll
		for(uint32_t a=0u; a<3u; a++) {
			F[(uint64_t)a*count+k] = v[a];
			float mean = acc[(uint64_t)a*count+k];
			const float d = __fsub_rn(v[a], mean);
			mean = __fadd_rn(mean, __fmul_rn(d, inv_n));
			acc[(uint64_t)a*count+k] = mean;
			acc[(uint64_t)(3u+a)*count+k] = __fadd_rn(acc[(uint64_t)(3u+a)*count+k], __fmul_rn(d, __fsub_rn(v[a], mean)));
		}
	}
}

// First level: partial[a*nchunks + h] = sum over the cells of chunk h (k in [chunk_begin[h], chunk_begin[h+1]), one label) of component a of (F, M), in index
// order, from +0.0. ref: r0 of every label [3*l + a]; chunk_label[h]: the label of chunk h.
__global__ void __launch_bounds__(256) k_wall_chunks(const __grid_constant__ DomainConst c, const uint64_t count, const uint64_t nchunks, const uint64_t* __restrict__ chunk_begin,
	const uint32_t* __restrict__ chunk_label, const uint64_t* __restrict__ cell, const float* __restrict__ F, const double* __restrict__ ref, double* __restrict__ partial) {
	for(uint64_t h=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; h<nchunks; h+=(uint64_t)gridDim.x*blockDim.x) {
		const uint32_t l = chunk_label[h];
		const double r0x = ref[3u*l], r0y = ref[3u*l+1u], r0z = ref[3u*l+2u];
		double s[WALL_COMPONENTS] = { 0.0, 0.0, 0.0, 0.0, 0.0, 0.0 };
		for(uint64_t k=chunk_begin[h]; k<chunk_begin[h+1u]; k++) {
			const uint64_t n = cell[k];
			const int x = (int)(n%c.Px)+c.Ox, y = (int)((n/c.Px)%c.Ny)+c.Oy, z = (int)(n/((uint64_t)c.Px*c.Ny))+c.Oz;
			const double fx = (double)F[k], fy = (double)F[count+k], fz = (double)F[2ull*count+k];
			const double dx = __dsub_rn((double)x, r0x), dy = __dsub_rn((double)y, r0y), dz = __dsub_rn((double)z, r0z);
			const double v[WALL_COMPONENTS] = { fx, fy, fz, __dsub_rn(__dmul_rn(dy, fz), __dmul_rn(dz, fy)), __dsub_rn(__dmul_rn(dz, fx), __dmul_rn(dx, fz)),
				__dsub_rn(__dmul_rn(dx, fy), __dmul_rn(dy, fx)) };
#pragma unroll
			for(uint32_t a=0u; a<WALL_COMPONENTS; a++) s[a] = __dadd_rn(s[a], v[a]);
		}
#pragma unroll
		for(uint32_t a=0u; a<WALL_COMPONENTS; a++) partial[(uint64_t)a*nchunks+h] = s[a];
	}
}

// Second and third level: segmented sums in order, one thread per (segment, component): out[s*os + a*oa] = the sum of in[a*nin + h] over
// begin[s] <= h < begin[s+1], from +0.0 (an empty segment gives 0). Second level: groups of up to WALL_GROUP consecutive chunks of one label; third level:
// the groups of every label, written to one sample of the ring [l*6 + a].
__global__ void __launch_bounds__(256) k_wall_segments(const uint64_t nseg, const uint64_t* __restrict__ begin, const uint64_t nin, const double* __restrict__ in,
	const uint64_t os, const uint64_t oa, double* __restrict__ out) {
	for(uint64_t q=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; q<nseg*WALL_COMPONENTS; q+=(uint64_t)gridDim.x*blockDim.x) {
		const uint64_t sg = q/WALL_COMPONENTS, a = q%WALL_COMPONENTS;
		double s = 0.0;
		for(uint64_t h=begin[sg]; h<begin[sg+1u]; h++) s = __dadd_rn(s, in[a*nin+h]);
		out[sg*os+a*oa] = s;
	}
}

} // namespace luw
