// Lagrangian tracer particles on the device: released from box emitters into a ring of slots, advected by the velocity read from the DDFs (no update_fields
// over the lattice, nothing written into it), with an optional uniform random walk for subgrid diffusion, and binned into concentration counts.
// The reference compiles its particle extension out (PARTICLES, integrate_particles in FX/kernel.cpp): there particles are float32, move with the
// trilinearly interpolated stored u, and may couple back to the fluid (IBM). Here positions are float64 (at x ~ 1000 a float32 ulp of 6e-5 cells
// swallows a near-wall move of 1e-3 cells per step), u is what update_fields + a read would give (probe_cell, lbm_probes.cuh), there is no back-coupling,
// and every float / double operation of the particle arithmetic is explicitly rounded (__fmul_rn ...), so that the STRICT and FAST builds differ only
// in the cell velocities. oracle/particles_oracle.py restates the model.
//  * position p: global = local lattice coordinates (single domains only), cell centres at integers;
//  * u(p): trilinear in float32 over the 8 cells around p: x0 = floor(p), clamped to N-2 on a non-periodic axis, x1 = x0+1 (wrapped on a periodic one),
//    f = (float)(p - x0); along x on the four edges, then y, then z, each a*(1-f) + b*f;
//  * move: p' = p + (double)u*(double)dt + sigma*sqrt(3)*(2U-1) per axis, U = (r >> 11)*2^-53 from Philox4x64-10 (counter (slot, call, 0, 0), key (seed, 0));
//    periodic axes wrap into [0, N); outside [0, N-1] on a non-periodic axis (or not finite) -> LEFT at p'; nearest cell floor(p'+0.5) solid -> wall mode 0
//    keeps p, wall mode 1 -> DEPOSITED at p';
//  * emit: slot (head+i) mod capacity, i = e*per + k, at c_e + h_e*(2U-1) per axis (counter (slot, call, 1, 0)), BURIED in a solid cell, ACTIVE otherwise;
//  * count: bins[(iz*By + iy)*Bx + ix] += 1 for every ACTIVE particle, i = floor(p+0.5) / b per axis.
#pragma once
#include "lbm_probes.cuh"

namespace luw {

enum : uint8_t { PT_FREE = 0u, PT_ACTIVE = 1u, PT_DEPOSITED = 2u, PT_LEFT = 3u, PT_BURIED = 4u };

struct ParticleSet { // device arrays of one particle ring and its fixed settings
	double* p; // SoA [3][capacity]
	uint8_t* state; uint32_t* emitter; uint64_t* release;
	uint64_t capacity, seed;
	uint32_t periodic, wall_mode; // periodic: bit a for axis a
};

// Philox4x64-10 (Salmon et al., SC'11; Random123's philox4x64 with 10 rounds): one block of 4 outputs for a 256-bit counter and a 128-bit key.
// numpy's np.random.Philox is the same generator; it increments its counter before producing a block.
__host__ __device__ inline void philox4x64_10(const uint64_t ctr[4], const uint64_t key[2], uint64_t out[4]) {
	uint64_t x0 = ctr[0], x1 = ctr[1], x2 = ctr[2], x3 = ctr[3], k0 = key[0], k1 = key[1];
	for(int r=0; r<10; r++) {
		const uint64_t m0 = 0xD2E7470EE14C6C93ull, m1 = 0xCA5A826395121157ull;
#ifdef __CUDA_ARCH__
		const uint64_t hi0 = __umul64hi(m0, x0), hi1 = __umul64hi(m1, x2);
#else
		const uint64_t hi0 = (uint64_t)(((unsigned __int128)m0*x0)>>64), hi1 = (uint64_t)(((unsigned __int128)m1*x2)>>64);
#endif
		const uint64_t lo0 = m0*x0, lo1 = m1*x2;
		x0 = hi1^x1^k0; x1 = lo1; x2 = hi0^x3^k1; x3 = lo0;
		k0 += 0x9E3779B97F4A7C15ull; k1 += 0xBB67AE8584CAA73Bull;
	}
	out[0] = x0; out[1] = x1; out[2] = x2; out[3] = x3;
}

namespace {

__device__ __forceinline__ double pt_uniform(const uint64_t r) { return __dmul_rn((double)(r>>11), 0x1.0p-53); } // [0, 1) on the 2^-53 grid
__device__ __forceinline__ double pt_sym(const uint64_t r) { return __dadd_rn(__dmul_rn(2.0, pt_uniform(r)), -1.0); } // 2U-1, exact
// q into [0, N) on a periodic axis; a non-finite q stays non-finite
__device__ __forceinline__ double pt_wrap(double q, const double N) {
	if(q>=0.0&&q<N) return q;
	q = __dadd_rn(q, -__dmul_rn(floor(__ddiv_rn(q, N)), N));
	if(q<0.0) q = __dadd_rn(q, N);
	if(q>=N) q = __dadd_rn(q, -N);
	return q;
}
// index of the cell nearest to q on an axis of N cells (q inside the lattice: [0, N) periodic, [0, N-1] otherwise)
__device__ __forceinline__ uint32_t pt_nearest(const double q, const uint32_t N) {
	const uint32_t k = (uint32_t)floor(__dadd_rn(q, 0.5));
	return k>=N ? k-N : k;
}
__device__ __forceinline__ bool pt_solid(const DomainConst& c, const double q[3]) {
	const uint64_t n = (uint64_t)pt_nearest(q[0], c.Nx)+((uint64_t)pt_nearest(q[1], c.Ny)+(uint64_t)pt_nearest(q[2], c.Nz)*c.Ny)*c.Px;
	return (c.flags[n]&TYPE_BO)==TYPE_S;
}
__device__ __forceinline__ float pt_lerp(const float a, const float b, const float f) { return __fadd_rn(__fmul_rn(a, __fadd_rn(1.0f, -f)), __fmul_rn(b, f)); }

} // anonymous namespace

namespace {

// one thread per slot, grid-stride; only ACTIVE particles move. call: this ring's advance count (the Philox counter's second word).
template<int P, uint32_t FEAT, bool TH> __global__ void __launch_bounds__(256) k_particles_advance(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a,
	const __grid_constant__ ParticleSet s, const uint64_t call, const float dt, const double sigma) {
	const uint32_t Nd[3] = { c.Nx, c.Ny, c.Nz };
	const double amp = __dmul_rn(sigma, 1.7320508075688772); // sigma*sqrt(3): half-width of the uniform step of variance sigma^2
	const uint64_t key[2] = { s.seed, 0ull };
	for(uint64_t k=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; k<s.capacity; k+=(uint64_t)gridDim.x*blockDim.x) {
		if(s.state[k]!=PT_ACTIVE) continue;
		double p[3];
		uint32_t lo[3], hi[3];
		float f[3];
		for(int d=0; d<3; d++) {
			p[d] = s.p[(uint64_t)d*s.capacity+k];
			const bool per = (s.periodic>>d)&1u;
			uint32_t x0 = (uint32_t)floor(p[d]);
			if(!per&&x0>Nd[d]-2u) x0 = Nd[d]-2u;
			lo[d] = x0; hi[d] = (per&&x0+1u==Nd[d]) ? 0u : x0+1u;
			f[d] = __double2float_rn(__dadd_rn(p[d], -(double)x0));
		}
		// corner k: x = k&1, y = (k>>1)&1, z = k>>2; edges along x first (even k: left end), then y (k&3 == 3), then z (k == 7)
		float ex[3] = { 0.0f, 0.0f, 0.0f }, ey[3] = { 0.0f, 0.0f, 0.0f }, ez[3] = { 0.0f, 0.0f, 0.0f }, u[3] = { 0.0f, 0.0f, 0.0f };
#pragma unroll 1
		for(uint32_t q=0u; q<8u; q++) {
			const uint64_t n = (uint64_t)((q&1u) ? hi[0] : lo[0])+((uint64_t)((q&2u) ? hi[1] : lo[1])+(uint64_t)((q&4u) ? hi[2] : lo[2])*c.Ny)*c.Px;
			float r_, v[3], T_;
			probe_cell<P, FEAT, TH>(c, a, n, r_, v[0], v[1], v[2], T_);
			(void)r_; (void)T_;
			for(int d=0; d<3; d++) {
				if(!(q&1u)) { ex[d] = v[d]; continue; }
				const float e = pt_lerp(ex[d], v[d], f[0]);
				if(!(q&2u)) { ey[d] = e; continue; }
				const float g = pt_lerp(ey[d], e, f[1]);
				if(!(q&4u)) ez[d] = g;
				else u[d] = pt_lerp(ez[d], g, f[2]);
			}
		}
		const uint64_t ctr[4] = { k, call, 0ull, 0ull };
		uint64_t r[4];
		philox4x64_10(ctr, key, r);
		double q[3];
		bool left = false;
		for(int d=0; d<3; d++) {
			q[d] = __dadd_rn(__dadd_rn(p[d], __dmul_rn((double)u[d], (double)dt)), __dmul_rn(amp, pt_sym(r[d])));
			const double N = (double)Nd[d];
			if((s.periodic>>d)&1u) { q[d] = pt_wrap(q[d], N); left |= !(q[d]>=0.0&&q[d]<N); }
			else left |= !(q[d]>=0.0&&q[d]<=N-1.0);
		}
		uint8_t st = PT_ACTIVE;
		if(left) st = PT_LEFT;
		else if(pt_solid(c, q)) {
			if(s.wall_mode==0u) continue; // rejected: the particle stays at p
			st = PT_DEPOSITED;
		}
		for(int d=0; d<3; d++) s.p[(uint64_t)d*s.capacity+k] = q[d];
		if(st!=PT_ACTIVE) s.state[k] = st;
	}
}

#ifndef LUW_PARTICLES_ADVANCE_ONLY
// release of E*per particles into slots head, head+1, ... (mod capacity) in the order [emitter][i]; box[6e..6e+5] = centre, half-extents. call: this ring's
// emit count. Emitter boxes lie inside [0, N-1] on non-periodic axes (luw_particles_create checks it).
__global__ void __launch_bounds__(256) k_particles_emit(const __grid_constant__ DomainConst c, const __grid_constant__ ParticleSet s, const double* __restrict__ box,
	const uint32_t per, const uint64_t total, const uint64_t head, const uint64_t call, const uint64_t t) {
	const uint32_t Nd[3] = { c.Nx, c.Ny, c.Nz };
	const uint64_t key[2] = { s.seed, 0ull };
	for(uint64_t i=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; i<total; i+=(uint64_t)gridDim.x*blockDim.x) {
		const uint64_t k = (head+i)%s.capacity;
		const uint32_t e = (uint32_t)(i/per);
		const uint64_t ctr[4] = { k, call, 1ull, 0ull };
		uint64_t r[4];
		philox4x64_10(ctr, key, r);
		double q[3];
		for(int d=0; d<3; d++) {
			q[d] = __dadd_rn(box[6u*e+d], __dmul_rn(box[6u*e+3u+d], pt_sym(r[d])));
			if((s.periodic>>d)&1u) q[d] = pt_wrap(q[d], (double)Nd[d]);
			s.p[(uint64_t)d*s.capacity+k] = q[d];
		}
		s.state[k] = pt_solid(c, q) ? PT_BURIED : PT_ACTIVE;
		s.emitter[k] = e;
		s.release[k] = t;
	}
}

// concentration counts: bin (ix, iy, iz) = nearest cell / bin size per axis; integer atomics, so the result does not depend on the order
__global__ void __launch_bounds__(256) k_particles_count(const __grid_constant__ DomainConst c, const __grid_constant__ ParticleSet s,
	const uint32_t bx, const uint32_t by, const uint32_t bz, const uint32_t Bx, const uint32_t By, uint32_t* __restrict__ bins) {
	for(uint64_t k=(uint64_t)blockIdx.x*blockDim.x+threadIdx.x; k<s.capacity; k+=(uint64_t)gridDim.x*blockDim.x) {
		if(s.state[k]!=PT_ACTIVE) continue;
		const uint32_t ix = pt_nearest(s.p[k], c.Nx)/bx, iy = pt_nearest(s.p[s.capacity+k], c.Ny)/by, iz = pt_nearest(s.p[2ull*s.capacity+k], c.Nz)/bz;
		atomicAdd(&bins[((uint64_t)iz*By+iy)*Bx+ix], 1u);
	}
}
#endif

} // anonymous namespace
} // namespace luw
