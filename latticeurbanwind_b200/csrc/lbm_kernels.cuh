// LBM kernels, generic one-cell-per-thread form (sm_100a). This file is compiled twice (lbm_strict.cu with -fmad=false,
// lbm_fast.cu with contraction) -- see LUW_ARITH_* in include/luw_cuda.h. The generic kernels are the always-correct path for
// every grid shape and flag pattern; lbm_tile.cuh / lbm_lean.cuh hold the TMA-staged two-cells-per-thread kernels that run wherever the lattice allows.
#pragma once
#include "lbm_common.cuh"

namespace luw {
namespace {

// ------------------------------------------------------------------ Esoteric-Pull load / store (FX/kernel.cpp:1338-1351)
template<int P> __device__ __forceinline__ void load_f(const typename Ddf<P>::T* __restrict__ fi, const uint64_t N, const uint64_t* j, const uint32_t odd, float* f) {
	f[0] = Ddf<P>::dec(fi[j[0]]);
#pragma unroll
	for(uint32_t i=1u; i<Q; i+=2u) {
		f[i   ] = Ddf<P>::dec(fi[(uint64_t)(odd ? i    : i+1u)*N+j[0]]);
		f[i+1u] = Ddf<P>::dec(fi[(uint64_t)(odd ? i+1u : i   )*N+j[i]]);
	}
}
template<int P> __device__ __forceinline__ void store_f(typename Ddf<P>::T* __restrict__ fi, const uint64_t N, const uint64_t* j, const uint32_t odd, const float* f) {
	fi[j[0]] = Ddf<P>::enc(f[0]);
#pragma unroll
	for(uint32_t i=1u; i<Q; i+=2u) {
		fi[(uint64_t)(odd ? i+1u : i   )*N+j[i]] = Ddf<P>::enc(f[i   ]);
		fi[(uint64_t)(odd ? i    : i+1u)*N+j[0]] = Ddf<P>::enc(f[i+1u]);
	}
}

// ------------------------------------------------------------------ the collision of one cell, shared by the generic and the pair kernels' slow path
// in: streamed DDFs f[19]; out: post-collision f[19]; writes rho/u when UPDATE_FIELDS (FX/kernel.cpp:1503-1748)
template<uint32_t FEAT> __device__ __forceinline__ void collide_cell(const DomainConst& c, const StepArgs& a, const uint64_t n,
	const uint32_t x, const uint32_t y, const uint32_t z, const uint32_t bo, float* f) {
	constexpr bool UF = (FEAT&F_UPDATE_FIELDS)!=0u, VF = (FEAT&F_VOLUME_FORCE)!=0u, EQ = (FEAT&F_EQUILIBRIUM)!=0u, SG = (FEAT&F_SUBGRID)!=0u;
	const bool is_e = EQ&&bo==TYPE_E;
	float rhon, uxn, uyn, uzn;
	if(is_e) { rhon = c.rho[n]; uxn = c.u[n]; uyn = c.u[c.N+n]; uzn = c.u[2ull*c.N+n]; }
	else rho_u(f, rhon, uxn, uyn, uzn);
	float Fin[Q];
	if(VF) {
		float fxn, fyn, fzn;
		luw_force(c, a, x, y, z, bo, true, rhon, uxn, uyn, uzn, fxn, fyn, fzn);
		const float rho2 = 0.5f/rhon;
		uxn = clampc(fmaf(fxn, rho2, uxn)); uyn = clampc(fmaf(fyn, rho2, uyn)); uzn = clampc(fmaf(fzn, rho2, uzn));
		forcing_terms(uxn, uyn, uzn, fxn, fyn, fzn, Fin);
	} else {
		uxn = clampc(uxn); uyn = clampc(uyn); uzn = clampc(uzn);
	}
	if(UF&&!is_e) { c.rho[n] = rhon; c.u[n] = uxn; c.u[c.N+n] = uyn; c.u[2ull*c.N+n] = uzn; }
	float feq[Q];
	f_eq(rhon, uxn, uyn, uzn, feq);
	float w = c.w;
	if(SG) w = smagorinsky_w(w, f, feq, rhon);
	if(is_e) {
#pragma unroll
		for(int i=0; i<Q; i++) f[i] = feq[i];
	} else if(VF) {
		const float c_tau = fmaf(w, -0.5f, 1.0f), omw = 1.0f-w;
#pragma unroll
		for(int i=0; i<Q; i++) f[i] = fmaf(omw, f[i], fmaf(w, feq[i], Fin[i]*c_tau));
	} else {
		const float omw = 1.0f-w;
#pragma unroll
		for(int i=0; i<Q; i++) f[i] = fmaf(omw, f[i], fmaf(w, feq[i], 0.0f));
	}
}

// ------------------------------------------------------------------ kernel: stream_collide (FX/kernel.cpp:1475-1780), one cell per thread
template<int P, uint32_t FEAT> __global__ void __launch_bounds__(128) k_stream_collide(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a) {
	typedef typename Ddf<P>::T T;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const uint64_t n = j[0];
	const uint32_t fl = c.flags[n], bo = fl&TYPE_BO;
	if(bo==TYPE_S||(fl&TYPE_SU)==TYPE_G) return;
	const uint32_t odd = (uint32_t)(a.t&1ull);
	float f[Q];
	load_f<P>((const T*)c.fi, c.N, j, odd, f);
	collide_cell<FEAT>(c, a, n, x, y, z, bo, f);
	store_f<P>((T*)c.fi, c.N, j, odd, f);
}

// ------------------------------------------------------------------ kernel: initialize (FX/kernel.cpp:1370-1452)
template<int P> __global__ void __launch_bounds__(128) k_initialize(const __grid_constant__ DomainConst c) {
	typedef typename Ddf<P>::T T;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const uint64_t n = j[0];
	if((c.flags[n]&TYPE_BO)==TYPE_S) { c.u[n] = 0.0f; c.u[c.N+n] = 0.0f; c.u[2ull*c.N+n] = 0.0f; }
	float feq[Q];
	f_eq(c.rho[n], c.u[n], c.u[c.N+n], c.u[2ull*c.N+n], feq);
	store_f<P>((T*)c.fi, c.N, j, 1u, feq);
}

// ------------------------------------------------------------------ halo kernels (FX/kernel.cpp:2188-2297)
__constant__ uint8_t XFER[6][5] = { // index_transfer(), D3Q19: the 5 DDFs that cross each face
	{1, 7,13, 9,15}, {2, 8,14,10,16}, {3, 7,14,11,17}, {4, 8,13,12,18}, {5, 9,16,11,18}, {6,10,15,12,17}
};
// thread index t of a face of axis d on layer `layer` -> cell (x,y,z) and payload index a. The reference numbers face cells like index_extract_p/m
// (FX/kernel.cpp:2192-2207): x: a=y+z*Ny, y: a=z+x*Nz, z: a=x+y*Nx. Threads always run x-fastest where the face has an x extent, so that lattice
// accesses coalesce (the reference's y-face order walks z fastest: a stride of Nx*Ny elements per thread, measured 2.4x slower than a z face of the same area);
// `xfast` also lays the payload out in thread order -- for buffers that only this library reads (in-process and IPC exchanges).
__device__ __forceinline__ void face_xyz(const DomainConst& c, const uint32_t d, const uint32_t t, const uint32_t layer, const bool xfast, uint32_t& x, uint32_t& y, uint32_t& z, uint32_t& a) {
	if(d==0u) { x = layer; y = t%c.Ny; z = t/c.Ny; a = t; }
	else if(d==1u) { x = t%c.Nx; y = layer; z = t/c.Nx; a = xfast ? t : z+x*c.Nz; }
	else { x = t%c.Nx; y = t/c.Nx; z = layer; a = t; }
}
__device__ __forceinline__ uint32_t axis_len(const DomainConst& c, const uint32_t d) { return d==0u ? c.Nx : d==1u ? c.Ny : c.Nz; }

// raw fpxx copies, no conversion. Faces normal to y / z: one thread per (face cell, side), blockIdx.y = side. Faces normal to x: one thread per face cell does
// BOTH sides -- the two face cells of a row (x = 1 / Nx-2, or 0 / Nx-1) lie in the same 1 KB lattice row of every slot, and touching them back to back lets
// the second access find the DRAM page the first one opened (every x-face element is a 2-byte access in its own row otherwise).
template<typename T, bool INSERT> __device__ __forceinline__ void halo_fi_cell(const DomainConst& c, const uint32_t d, const uint32_t A, const uint32_t odd, const bool xfast, const uint32_t t, const uint32_t side, T* __restrict__ buf) {
	const uint32_t L = axis_len(c, d);
	uint32_t x, y, z, a;
	face_xyz(c, d, t, INSERT ? (side==0u ? L-1u : 0u) : (side==0u ? L-2u : 1u), xfast, x, y, z, a);
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	T* fi = (T*)c.fi;
#pragma unroll
	for(uint32_t b=0u; b<5u; b++) {
		const uint32_t i = XFER[2u*d+side][b];
		if(INSERT) {
			const uint64_t cell = (i&1u) ? j[0] : j[i-1u];
			const uint32_t slot = odd ? i : ((i&1u) ? i+1u : i-1u);
			fi[(uint64_t)slot*c.N+cell] = buf[(uint64_t)b*A+a];
		} else {
			const uint64_t cell = (i&1u) ? j[i] : j[0];
			const uint32_t slot = odd ? ((i&1u) ? i+1u : i-1u) : i;
			buf[(uint64_t)b*A+a] = fi[(uint64_t)slot*c.N+cell];
		}
	}
}
template<typename T, bool INSERT> __global__ void __launch_bounds__(128) k_halo_fi(const __grid_constant__ DomainConst c, const uint32_t d, const uint32_t A, const uint32_t odd, const bool xfast, T* __restrict__ buf_p, T* __restrict__ buf_m) {
	const uint32_t t = blockIdx.x*blockDim.x+threadIdx.x;
	if(t>=A) return;
	if(gridDim.y==1u) { halo_fi_cell<T, INSERT>(c, d, A, odd, xfast, t, 0u, buf_p); halo_fi_cell<T, INSERT>(c, d, A, odd, xfast, t, 1u, buf_m); }
	else halo_fi_cell<T, INSERT>(c, d, A, odd, xfast, t, blockIdx.y, blockIdx.y==0u ? buf_p : buf_m);
}
template<bool INSERT> __device__ __forceinline__ void halo_ruf_cell(const DomainConst& c, const uint32_t d, const uint32_t A, const bool xfast, const uint32_t t, const uint32_t side, char* __restrict__ buf) {
	const uint32_t L = axis_len(c, d);
	uint32_t x, y, z, a;
	face_xyz(c, d, t, INSERT ? (side==0u ? L-1u : 0u) : (side==0u ? L-2u : 1u), xfast, x, y, z, a);
	const uint64_t n = x+((uint64_t)y+(uint64_t)z*c.Ny)*c.Px;
	float* bf = (float*)buf;
	uint8_t* bb = (uint8_t*)buf+16ull*A;
	if(INSERT) { c.rho[n] = bf[a]; c.u[n] = bf[(uint64_t)A+a]; c.u[c.N+n] = bf[2ull*A+a]; c.u[2ull*c.N+n] = bf[3ull*A+a]; c.flags[n] = bb[a]; }
	else { bf[a] = c.rho[n]; bf[(uint64_t)A+a] = c.u[n]; bf[2ull*A+a] = c.u[c.N+n]; bf[3ull*A+a] = c.u[2ull*c.N+n]; bb[a] = c.flags[n]; }
}
template<bool INSERT> __global__ void __launch_bounds__(128) k_halo_rho_u_flags(const __grid_constant__ DomainConst c, const uint32_t d, const uint32_t A, const bool xfast, char* __restrict__ buf_p, char* __restrict__ buf_m) {
	const uint32_t t = blockIdx.x*blockDim.x+threadIdx.x;
	if(t>=A) return;
	if(gridDim.y==1u) { halo_ruf_cell<INSERT>(c, d, A, xfast, t, 0u, buf_p); halo_ruf_cell<INSERT>(c, d, A, xfast, t, 1u, buf_m); }
	else halo_ruf_cell<INSERT>(c, d, A, xfast, t, blockIdx.y, blockIdx.y==0u ? buf_p : buf_m);
}

// ================================================================== thermal D3Q7 extension (TEMPERATURE), SURVEY.md 8-f4
// Correctness-first form: the one-cell-per-thread kernels with the reference's TEMPERATURE blocks fused in (the temperature collision needs the cell's velocity
// BEFORE the force half-step, which is never stored, so the g update has to live inside the momentum kernel: FX/kernel.cpp:1639-1684). The first seven
// entries of the D3Q19 neighbour list are exactly neighbors_temperature()'s j7 (FX/kernel.cpp:1307-1314).
__device__ __forceinline__ void g_eq(const float T, const float ux, const float uy, const float uz, float* geq) { // FX/kernel.cpp:1315-1321
	const float wsT4 = 0.5f*T, wsTm1 = 0.125f*(T-1.0f);
	geq[0] = fmaf(0.25f, T, -0.25f);
	geq[1] = fmaf(wsT4, ux, wsTm1); geq[2] = fmaf(wsT4, -ux, wsTm1);
	geq[3] = fmaf(wsT4, uy, wsTm1); geq[4] = fmaf(wsT4, -uy, wsTm1);
	geq[5] = fmaf(wsT4, uz, wsTm1); geq[6] = fmaf(wsT4, -uz, wsTm1);
}
template<int P> __device__ __forceinline__ void load_g(const typename Ddf<P>::T* gi, const uint64_t N, const uint64_t* j, const uint32_t odd, float* g) { // FX/kernel.cpp:1322-1328
	g[0] = Ddf<P>::dec(gi[j[0]]);
#pragma unroll
	for(uint32_t i=1u; i<7u; i+=2u) {
		g[i   ] = Ddf<P>::dec(gi[(uint64_t)(odd ? i    : i+1u)*N+j[0]]);
		g[i+1u] = Ddf<P>::dec(gi[(uint64_t)(odd ? i+1u : i   )*N+j[i]]);
	}
}
template<int P> __device__ __forceinline__ void store_g(typename Ddf<P>::T* gi, const uint64_t N, const uint64_t* j, const uint32_t odd, const float* g) { // FX/kernel.cpp:1329-1335
	gi[j[0]] = Ddf<P>::enc(g[0]);
#pragma unroll
	for(uint32_t i=1u; i<7u; i+=2u) {
		gi[(uint64_t)(odd ? i+1u : i   )*N+j[i]] = Ddf<P>::enc(g[i   ]);
		gi[(uint64_t)(odd ? i    : i+1u)*N+j[0]] = Ddf<P>::enc(g[i+1u]);
	}
}
// temperature of the cell from the streamed-in g (or the preset of a TYPE_T cell)
__device__ __forceinline__ float temperature_of(const DomainConst& c, const uint64_t n, const bool is_t, const float* g) {
	if(is_t) return c.T[n];
	float Tn = 0.0f;
#pragma unroll
	for(int i=0; i<7; i++) Tn += g[i];
	return Tn+1.0f; // 1 is added last (DDF shifting)
}
// stream_collide with the TEMPERATURE block: collide_cell's sequence (kept textually parallel to it) with the g update between the force assembly and
// the force half-step. Returns the post-collision f; g is streamed out here.
template<int P, uint32_t FEAT> __device__ __forceinline__ void collide_cell_thermal(const DomainConst& c, const StepArgs& a, const uint64_t* j,
	const uint32_t x, const uint32_t y, const uint32_t z, const uint32_t fl, const uint32_t odd, float* f) {
	typedef typename Ddf<P>::T S;
	constexpr bool UF = (FEAT&F_UPDATE_FIELDS)!=0u, VF = (FEAT&F_VOLUME_FORCE)!=0u, EQ = (FEAT&F_EQUILIBRIUM)!=0u, SG = (FEAT&F_SUBGRID)!=0u;
	const uint64_t n = j[0];
	const uint32_t bo = fl&TYPE_BO;
	const bool is_e = EQ&&bo==TYPE_E, is_t = (fl&TYPE_T)!=0u;
	float rhon, uxn, uyn, uzn;
	if(is_e) { rhon = c.rho[n]; uxn = c.u[n]; uyn = c.u[c.N+n]; uzn = c.u[2ull*c.N+n]; }
	else rho_u(f, rhon, uxn, uyn, uzn);
	// ---- TEMPERATURE block, FX/kernel.cpp:1639-1684
	float g[7];
	load_g<P>((const S*)c.gi, c.N, j, odd, g);
	float Tn = temperature_of(c, n, is_t, g);
	if((c.features&F_SPONGE)&&!is_t&&bo!=TYPE_E&&c.has_t) { // sponge on T towards the top row of the column (def_sponge_ref_mode 0)
		const int dt = (int)(c.Nzg-2u)-((int)z+c.Oz);
		if(dt>=0&&dt<(int)c.sponge_N) {
			const float sg = __ldg(c.sigma+dt);
			const uint64_t nref = (uint64_t)x+((uint64_t)y+(uint64_t)c.tz*c.Ny)*c.Px;
			Tn = fmaf(sg, c.T[nref]-Tn, Tn); // plain load: T is written by this kernel (the top row itself is TYPE_T / TYPE_E in LUW's decks)
		}
	}
	float geq[7];
	g_eq(Tn, uxn, uyn, uzn, geq); // velocity BEFORE the force half-step
	if(is_t) {
#pragma unroll
		for(int i=0; i<7; i++) g[i] = geq[i];
	} else {
		if(UF) c.T[n] = Tn;
		const float omw_T = 1.0f-c.w_T;
#pragma unroll
		for(int i=0; i<7; i++) g[i] = fmaf(omw_T, g[i], c.w_T*geq[i]);
	}
	store_g<P>((S*)c.gi, c.N, j, odd, g);
	// ---- momentum, as collide_cell
	float Fin[Q];
	if(VF) {
		float fxn, fyn, fzn;
		luw_force(c, a, x, y, z, bo, true, rhon, uxn, uyn, uzn, fxn, fyn, fzn);
		const float dT = Tn-c.T_avg; // buoyancy (Boussinesq); LUW runs with f = 0
		fxn -= a.fx*c.beta*dT; fyn -= a.fy*c.beta*dT; fzn -= a.fz*c.beta*dT;
		const float rho2 = 0.5f/rhon;
		uxn = clampc(fmaf(fxn, rho2, uxn)); uyn = clampc(fmaf(fyn, rho2, uyn)); uzn = clampc(fmaf(fzn, rho2, uzn));
		forcing_terms(uxn, uyn, uzn, fxn, fyn, fzn, Fin);
	} else {
		uxn = clampc(uxn); uyn = clampc(uyn); uzn = clampc(uzn);
	}
	if(UF&&!is_e) { c.rho[n] = rhon; c.u[n] = uxn; c.u[c.N+n] = uyn; c.u[2ull*c.N+n] = uzn; }
	float feq[Q];
	f_eq(rhon, uxn, uyn, uzn, feq);
	float w = c.w;
	if(SG) w = smagorinsky_w(w, f, feq, rhon);
	if(is_e) {
#pragma unroll
		for(int i=0; i<Q; i++) f[i] = feq[i];
	} else if(VF) {
		const float c_tau = fmaf(w, -0.5f, 1.0f), omw = 1.0f-w;
#pragma unroll
		for(int i=0; i<Q; i++) f[i] = fmaf(omw, f[i], fmaf(w, feq[i], Fin[i]*c_tau));
	} else {
		const float omw = 1.0f-w;
#pragma unroll
		for(int i=0; i<Q; i++) f[i] = fmaf(omw, f[i], fmaf(w, feq[i], 0.0f));
	}
}
template<int P, uint32_t FEAT> __global__ void __launch_bounds__(128) k_stream_collide_thermal(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a) {
	typedef typename Ddf<P>::T T;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const uint64_t n = j[0];
	const uint32_t fl = c.flags[n], bo = fl&TYPE_BO;
	if(bo==TYPE_S||(fl&TYPE_SU)==TYPE_G) return;
	const uint32_t odd = (uint32_t)(a.t&1ull);
	float f[Q];
	load_f<P>((const T*)c.fi, c.N, j, odd, f);
	collide_cell_thermal<P, FEAT>(c, a, j, x, y, z, fl, odd, f);
	store_f<P>((T*)c.fi, c.N, j, odd, f);
}
// The TEMPERATURE block alone (FX/kernel.cpp:1639-1684), second kernel of the two-kernel thermal step: the TMA-tiled momentum kernel has left every executing
// non-TYPE_E cell's velocity before the force half-step in c.upre (TYPE_E cells keep theirs in the boundary field c.u); the arithmetic is collide_cell_thermal's, line by
// line. Only legal while the buoyancy term vanishes (f = 0 or beta = 0, as in every LUW mode): with buoyancy the momentum step depends on this step's T, and
// enqueue_step runs the fused one-cell-per-thread kernel instead. FEAT: UPDATE_FIELDS (T is stored) and EQUILIBRIUM_BOUNDARIES matter.
template<int P, uint32_t FEAT> __global__ void __launch_bounds__(128) k_thermal_g(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a) {
	typedef typename Ddf<P>::T S;
	constexpr bool UF = (FEAT&F_UPDATE_FIELDS)!=0u, EQ = (FEAT&F_EQUILIBRIUM)!=0u;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j); // the first seven entries are neighbors_temperature()'s j7
	const uint64_t n = j[0];
	const uint32_t fl = c.flags[n], bo = fl&TYPE_BO;
	if(bo==TYPE_S||(fl&TYPE_SU)==TYPE_G) return;
	const uint32_t odd = (uint32_t)(a.t&1ull);
	const bool is_e = EQ&&bo==TYPE_E, is_t = (fl&TYPE_T)!=0u;
	const float* const us = is_e ? c.u : c.upre;
	const float uxn = us[n], uyn = us[c.N+n], uzn = us[2ull*c.N+n];
	float g[7];
	load_g<P>((const S*)c.gi, c.N, j, odd, g);
	float Tn = temperature_of(c, n, is_t, g);
	if((c.features&F_SPONGE)&&!is_t&&bo!=TYPE_E&&c.has_t) {
		const int dt = (int)(c.Nzg-2u)-((int)z+c.Oz);
		if(dt>=0&&dt<(int)c.sponge_N) {
			const float sg = __ldg(c.sigma+dt);
			const uint64_t nref = (uint64_t)x+((uint64_t)y+(uint64_t)c.tz*c.Ny)*c.Px;
			Tn = fmaf(sg, c.T[nref]-Tn, Tn);
		}
	}
	float geq[7];
	g_eq(Tn, uxn, uyn, uzn, geq);
	if(is_t) {
#pragma unroll
		for(int i=0; i<7; i++) g[i] = geq[i];
	} else {
		if(UF) c.T[n] = Tn;
		const float omw_T = 1.0f-c.w_T;
#pragma unroll
		for(int i=0; i<7; i++) g[i] = fmaf(omw_T, g[i], c.w_T*geq[i]);
	}
	store_g<P>((S*)c.gi, c.N, j, odd, g);
}
// initialize with the TEMPERATURE block (FX/kernel.cpp:1442-1450): g starts at g_eq(T, u)
template<int P> __global__ void __launch_bounds__(128) k_initialize_thermal(const __grid_constant__ DomainConst c) {
	typedef typename Ddf<P>::T T;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const uint64_t n = j[0];
	if((c.flags[n]&TYPE_BO)==TYPE_S) { c.u[n] = 0.0f; c.u[c.N+n] = 0.0f; c.u[2ull*c.N+n] = 0.0f; }
	const float uxn = c.u[n], uyn = c.u[c.N+n], uzn = c.u[2ull*c.N+n];
	float feq[Q];
	f_eq(c.rho[n], uxn, uyn, uzn, feq);
	float geq[7];
	g_eq(c.T[n], uxn, uyn, uzn, geq);
	store_g<P>((T*)c.gi, c.N, j, 1u, geq);
	store_f<P>((T*)c.fi, c.N, j, 1u, feq);
}
// ------------------------------------------------------------------ update_fields of one executing cell (FX/kernel.cpp:1938-2028; TEMPERATURE block 1981-2000)
// rho, u (and, TH, T) from the DDFs streamed in at a.t: no collision, no relaxation zones. The caller has skipped TYPE_S / TYPE_G cells and decides what is
// stored (TYPE_E keeps its boundary rho / u under EQUILIBRIUM_BOUNDARIES). k_update_fields, k_update_fields_thermal and k_probe_sample (lbm_probes.cuh) all
// compute through this function, so a probe equals update_fields bit for bit in either arithmetic build.
template<int P, uint32_t FEAT, bool TH> __device__ __forceinline__ void update_fields_cell(const DomainConst& c, const StepArgs& a, const uint64_t* j,
	const uint32_t x, const uint32_t y, const uint32_t z, const uint32_t fl, float& rhon, float& uxn, float& uyn, float& uzn, float& Tn) {
	typedef typename Ddf<P>::T T;
	constexpr bool VF = (FEAT&F_VOLUME_FORCE)!=0u;
	const uint32_t bo = fl&TYPE_BO, odd = (uint32_t)(a.t&1ull);
	float f[Q];
	load_f<P>((const T*)c.fi, c.N, j, odd, f);
	rho_u(f, rhon, uxn, uyn, uzn);
	if constexpr(TH) {
		float g[7];
		load_g<P>((const T*)c.gi, c.N, j, odd, g);
		Tn = temperature_of(c, j[0], (fl&TYPE_T)!=0u, g);
	}
	if(VF) {
		float fxn, fyn, fzn;
		luw_force(c, a, x, y, z, bo, false, rhon, uxn, uyn, uzn, fxn, fyn, fzn);
		if constexpr(TH) {
			const float dT = Tn-c.T_avg;
			fxn -= a.fx*c.beta*dT; fyn -= a.fy*c.beta*dT; fzn -= a.fz*c.beta*dT;
		}
		const float rho2 = 0.5f/rhon;
		uxn = clampc(fmaf(fxn, rho2, uxn)); uyn = clampc(fmaf(fyn, rho2, uyn)); uzn = clampc(fmaf(fzn, rho2, uzn));
	} else {
		uxn = clampc(uxn); uyn = clampc(uyn); uzn = clampc(uzn);
	}
}
// ------------------------------------------------------------------ kernel: update_fields (FX/kernel.cpp:1938-2028): no collision, no relaxation zones
template<int P, uint32_t FEAT> __global__ void __launch_bounds__(128) k_update_fields(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a) {
	constexpr bool EQ = (FEAT&F_EQUILIBRIUM)!=0u;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const uint64_t n = j[0];
	const uint32_t fl = c.flags[n], bo = fl&TYPE_BO;
	if(bo==TYPE_S||(fl&TYPE_SU)==TYPE_G) return;
	float rhon, uxn, uyn, uzn, Tn;
	update_fields_cell<P, FEAT, false>(c, a, j, x, y, z, fl, rhon, uxn, uyn, uzn, Tn);
	if(!(EQ&&bo==TYPE_E)) { c.rho[n] = rhon; c.u[n] = uxn; c.u[c.N+n] = uyn; c.u[2ull*c.N+n] = uzn; }
}
// update_fields with the TEMPERATURE block (FX/kernel.cpp:1981-2000): T from the streamed-in g, no sponge, no collision
template<int P, uint32_t FEAT> __global__ void __launch_bounds__(128) k_update_fields_thermal(const __grid_constant__ DomainConst c, const __grid_constant__ StepArgs a) {
	constexpr bool EQ = (FEAT&F_EQUILIBRIUM)!=0u;
	const uint32_t x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y, z = blockIdx.z;
	if(x>=c.Nx||is_halo(c, x, y, z)) return;
	uint64_t j[Q];
	neighbors(c, x, y, z, j);
	const uint64_t n = j[0];
	const uint32_t fl = c.flags[n], bo = fl&TYPE_BO;
	if(bo==TYPE_S||(fl&TYPE_SU)==TYPE_G) return;
	float rhon, uxn, uyn, uzn, Tn;
	update_fields_cell<P, FEAT, true>(c, a, j, x, y, z, fl, rhon, uxn, uyn, uzn, Tn);
	if(!(fl&TYPE_T)) c.T[n] = Tn;
	if(!(EQ&&bo==TYPE_E)) { c.rho[n] = rhon; c.u[n] = uxn; c.u[c.N+n] = uyn; c.u[2ull*c.N+n] = uzn; }
}
// halos of gi (one DDF per face cell and side: i = 2*axis+1 leaves through the + face, 2*axis+2 through the - face) and of T, FX/kernel.cpp:2337-2377
template<typename T, bool INSERT> __device__ __forceinline__ void halo_gi_cell(const DomainConst& c, const uint32_t d, const uint32_t odd, const bool xfast, const uint32_t t, const uint32_t side, T* __restrict__ buf) {
	const uint32_t L = axis_len(c, d);
	uint32_t x, y, z, a;
	face_xyz(c, d, t, INSERT ? (side==0u ? L-1u : 0u) : (side==0u ? L-2u : 1u), xfast, x, y, z, a);
	// the only neighbour either direction needs is the one a step along +axis (j7[2d+1]): extract reads it for the DDF leaving through the + face (odd i),
	// insert writes it for the DDF arriving through the - face (even i, j7[i-1]); no neighbour table, hence no local-memory array
	const uint64_t row = c.Px, plane = (uint64_t)c.Px*c.Ny;
	const uint64_t n = (uint64_t)x+y*row+z*plane;
	const uint32_t xp = d==0u ? (x+1u==c.Nx ? 0u : x+1u) : x, yp = d==1u ? (y+1u==c.Ny ? 0u : y+1u) : y, zp = d==2u ? (z+1u==c.Nz ? 0u : z+1u) : z;
	const uint64_t np = (uint64_t)xp+yp*row+zp*plane;
	T* gi = (T*)c.gi;
	const uint32_t i = 2u*d+side+1u;
	if(INSERT) {
		const uint64_t cell = (i&1u) ? n : np;
		const uint32_t slot = odd ? i : ((i&1u) ? i+1u : i-1u);
		gi[(uint64_t)slot*c.N+cell] = buf[a];
	} else {
		const uint64_t cell = (i&1u) ? np : n;
		const uint32_t slot = odd ? ((i&1u) ? i+1u : i-1u) : i;
		buf[a] = gi[(uint64_t)slot*c.N+cell];
	}
}
template<typename T, bool INSERT> __global__ void __launch_bounds__(128) k_halo_gi(const __grid_constant__ DomainConst c, const uint32_t d, const uint32_t A, const uint32_t odd, const bool xfast, T* __restrict__ buf_p, T* __restrict__ buf_m) {
	const uint32_t t = blockIdx.x*blockDim.x+threadIdx.x;
	if(t>=A) return;
	halo_gi_cell<T, INSERT>(c, d, odd, xfast, t, 0u, buf_p);
	halo_gi_cell<T, INSERT>(c, d, odd, xfast, t, 1u, buf_m);
}
template<bool INSERT> __global__ void __launch_bounds__(128) k_halo_T(const __grid_constant__ DomainConst c, const uint32_t d, const uint32_t A, const bool xfast, float* __restrict__ buf_p, float* __restrict__ buf_m) {
	const uint32_t t = blockIdx.x*blockDim.x+threadIdx.x;
	if(t>=A) return;
	const uint32_t L = axis_len(c, d);
#pragma unroll
	for(uint32_t side=0u; side<2u; side++) {
		uint32_t x, y, z, a;
		face_xyz(c, d, t, INSERT ? (side==0u ? L-1u : 0u) : (side==0u ? L-2u : 1u), xfast, x, y, z, a);
		const uint64_t n = x+((uint64_t)y+(uint64_t)z*c.Ny)*c.Px;
		float* buf = side==0u ? buf_p : buf_m;
		if(INSERT) c.T[n] = buf[a]; else buf[a] = c.T[n];
	}
}

// ------------------------------------------------------------------ kernel: vk_inlet_apply (FX/kernel.cpp:2495-2571)
// one thread per inlet point; the mode table (10 x V floats) is shared by all points of a face and stays L1/L2 resident
__global__ void __launch_bounds__(128) k_vk_inlet_apply(const uint64_t Ncells, const uint32_t use_interp, const float t0, const float t1, const float alpha,
	const uint64_t P, const uint64_t M, const uint64_t V, const uint64_t* __restrict__ point_cell, const uint8_t* __restrict__ point_face,
	const float* __restrict__ pd, const float* __restrict__ md, float* __restrict__ u) {
	const uint64_t i = (uint64_t)blockIdx.x*blockDim.x+threadIdx.x;
	if(i>=P) return;
	const uint64_t n = point_cell[i];
	const uint64_t fid = point_face[i]&0x07u;
	const float px = pd[i], py = pd[P+i], pz = pd[2ull*P+i];
	const float ubx = pd[3ull*P+i], uby = pd[4ull*P+i], ubz = pd[5ull*P+i], sigma = pd[6ull*P+i];
	if(fid>=5ull||!(sigma>0.0f)) { u[n] = ubx; u[Ncells+n] = uby; u[2ull*Ncells+n] = ubz; return; }
	float qx = 0.0f, qy = 0.0f, qz = 0.0f;
	for(uint64_t m=0ull; m<M; m++) {
		const uint64_t k = fid*M+m;
		const float kx = __ldg(md+k), ky = __ldg(md+V+k), kz = __ldg(md+2ull*V+k), om = __ldg(md+3ull*V+k);
		const float Ax = __ldg(md+4ull*V+k), Ay = __ldg(md+5ull*V+k), Az = __ldg(md+6ull*V+k);
		const float phx = __ldg(md+7ull*V+k), phy = __ldg(md+8ull*V+k), phz = __ldg(md+9ull*V+k);
		const float ph0 = fmaf(kx, px, fmaf(ky, py, fmaf(kz, pz, om*t0)));
		float vx = Ax*cosf(ph0+phx), vy = Ay*cosf(ph0+phy), vz = Az*cosf(ph0+phz);
		if(use_interp!=0u) {
			const float ph1 = fmaf(kx, px, fmaf(ky, py, fmaf(kz, pz, om*t1)));
			const float vx1 = Ax*cosf(ph1+phx), vy1 = Ay*cosf(ph1+phy), vz1 = Az*cosf(ph1+phz);
			vx = fmaf(alpha, vx1-vx, vx); vy = fmaf(alpha, vy1-vy, vy); vz = fmaf(alpha, vz1-vz, vz);
		}
		qx += vx; qy += vy; qz += vz;
	}
	u[n] = fmaf(sigma, qx, ubx); u[Ncells+n] = fmaf(sigma, qy, uby); u[2ull*Ncells+n] = fmaf(sigma, qz, ubz);
}

// ------------------------------------------------------------------ kernel: voxelize_mesh (FX/kernel.cpp:2381-2471), resting geometry
// One thread per column of the face normal to `direction`; the triangles are staged through shared memory in chunks that the whole block walks
// (the reference reads all of them from global memory per work-item). Ray/triangle arithmetic in the reference's operation order; this kernel is always
// taken from the STRICT translation unit (-fmad=false, IEEE division), because the flags must be bit-exact and a contracted product flips grazing rays.
struct VoxBox { uint32_t ntri; float x0, y0, z0, x1, y1, z1; };
struct VoxColumn { // one ray: the column it runs along, its origin, and what it has crossed so far
	uint32_t X, Y, Z;
	float rox, roy, roz, dx, dy, dz;
	bool out_of_box;
	uint32_t intersections, intersections_check;
	uint16_t distances[64];
};
// column (c0, c1) of the face normal to `direction`: (y, z) for x-rays, (z, x) for y-rays, (x, y) for z-rays -- the reference's a % n0, a / n0 (FX/kernel.cpp:2386-2393)
__device__ __forceinline__ void vox_column(const DomainConst& c, const uint32_t direction, const uint32_t c0, const uint32_t c1, const VoxBox& bb, VoxColumn& col) {
	const int Nx = (int)c.Nx, Ny = (int)c.Ny, Nz = (int)c.Nz;
	const auto clampi = [](const int x, const int lo, const int hi) { return x<lo ? lo : (x>hi ? hi : x); };
	if(direction==0u) { col.X = (uint32_t)clampi((int)bb.x0-c.Ox, 0, Nx-1); col.Y = c0; col.Z = c1; }
	else if(direction==1u) { col.X = c1; col.Y = (uint32_t)clampi((int)bb.y0-c.Oy, 0, Ny-1); col.Z = c0; }
	else { col.X = c0; col.Y = c1; col.Z = (uint32_t)clampi((int)bb.z0-c.Oz, 0, Nz-1); }
	const float offx = 0.5f*(float)(Nx+2*c.Ox)-0.5f, offy = 0.5f*(float)(Ny+2*c.Oy)-0.5f, offz = 0.5f*(float)(Nz+2*c.Oz)-0.5f;
	col.rox = ((float)col.X+0.5f-0.5f*(float)Nx)+offx; col.roy = ((float)col.Y+0.5f-0.5f*(float)Ny)+offy; col.roz = ((float)col.Z+0.5f-0.5f*(float)Nz)+offz;
	col.dx = (float)(direction==0u); col.dy = (float)(direction==1u); col.dz = (float)(direction==2u);
	const float rox = col.rox, roy = col.roy, roz = col.roz;
	col.out_of_box = direction==0u ? (roy<bb.y0||roz<bb.z0||roy>=bb.y1||roz>=bb.z1) : direction==1u ? (rox<bb.x0||roz<bb.z0||rox>=bb.x1||roz>=bb.z1) : (rox<bb.x0||roy<bb.y0||rox>=bb.x1||roy>=bb.y1);
	col.intersections = 0u; col.intersections_check = 0u;
}
// ray against the triangle (a, a+u.., a+v..) given as p0, p1, p2 (FX/kernel.cpp:2404-2423)
__device__ __forceinline__ void vox_cross(VoxColumn& col, const float ax, const float ay, const float az, const float bx, const float by, const float bz, const float cx, const float cy, const float cz) {
	const float dx = col.dx, dy = col.dy, dz = col.dz;
	const float ux = bx-ax, uy = by-ay, uz = bz-az;
	const float vx = cx-ax, vy = cy-ay, vz = cz-az;
	const float wx = col.rox-ax, wy = col.roy-ay, wz = col.roz-az;
	const float hx = dy*vz-dz*vy, hy = dz*vx-dx*vz, hz = dx*vy-dy*vx; // cross(r_direction, v)
	const float qx = wy*uz-wz*uy, qy = wz*ux-wx*uz, qz = wx*uy-wy*ux; // cross(w, u)
	const float g = ux*hx+uy*hy+uz*hz, f = 1.0f/g, s = f*(wx*hx+wy*hy+wz*hz), t = f*(dx*qx+dy*qy+dz*qz), d = f*(vx*qx+vy*qy+vz*qz);
	if(g!=0.0f&&s>=0.0f&&s<1.0f&&t>=0.0f&&s+t<1.0f) {
		if(d>0.0f) { if(col.intersections<64u&&d<65536.0f) col.distances[col.intersections] = (uint16_t)d; col.intersections++; }
		else col.intersections_check++;
	}
}
// the crossings sorted, the cells of the column between them flagged (FX/kernel.cpp:2425-2470)
__device__ __forceinline__ void vox_fill(const DomainConst& c, const uint32_t direction, const uint8_t flag, const VoxBox& bb, VoxColumn& col) {
	const int Nx = (int)c.Nx, Ny = (int)c.Ny, Nz = (int)c.Nz;
	const auto clampi = [](const int x, const int lo, const int hi) { return x<lo ? lo : (x>hi ? hi : x); };
	const uint32_t intersections = col.intersections, intersections_check = col.intersections_check, X = col.X, Y = col.Y, Z = col.Z;
	uint16_t* distances = col.distances;
	const uint32_t nsort = intersections<64u ? intersections : 64u;
	for(uint32_t i=1u; i<nsort; i++) { const uint16_t t = distances[i]; int j = (int)i-1; while(j>=0&&distances[j]>t) { distances[j+1] = distances[j]; j--; } distances[j+1] = t; }
	bool inside = (intersections%2u)&&(intersections_check%2u);
	uint32_t intersection = intersections%2u!=intersections_check%2u;
	const uint32_t h0 = direction==0u ? X : direction==1u ? Y : Z;
	const uint32_t hmax = direction==0u ? (uint32_t)clampi((int)bb.x1-c.Ox, 0, Nx) : direction==1u ? (uint32_t)clampi((int)bb.y1-c.Oy, 0, Ny) : (uint32_t)clampi((int)bb.z1-c.Oz, 0, Nz);
	const uint32_t hmesh = h0+(uint32_t)(intersections>0u ? distances[intersections-1u<63u ? intersections-1u : 63u] : 0u);
	for(uint32_t h=h0; h<hmax; h++) {
		while(intersection<intersections&&h>h0+(uint32_t)distances[intersection<63u ? intersection : 63u]) { inside = !inside; intersection++; }
		inside = inside&&(intersection<intersections&&h<hmesh);
		const uint64_t n = (uint64_t)(direction==0u ? h : X)+((uint64_t)(direction==1u ? h : Y)+(uint64_t)(direction==2u ? h : Z)*c.Ny)*c.Px;
		uint8_t fl = c.flags[n];
		if(inside) fl = (uint8_t)((fl&~TYPE_BO)|flag);
		else if((fl&TYPE_BO)==TYPE_S) { // previously solid, outside now: released if it carries the geometry's velocity (0 for resting geometry)
			if(c.u[n]==0.0f&&c.u[c.N+n]==0.0f&&c.u[2ull*c.N+n]==0.0f) fl = (uint8_t)(fl&~flag);
		}
		c.flags[n] = fl;
	}
}
__global__ void __launch_bounds__(128) k_voxelize_mesh(const __grid_constant__ DomainConst c, const uint32_t direction, const uint32_t A, const uint8_t flag, const VoxBox bb,
	const float* __restrict__ p0, const float* __restrict__ p1, const float* __restrict__ p2) {
	__shared__ float tri[128][9];
	const uint32_t a = blockIdx.x*blockDim.x+threadIdx.x;
	const uint32_t n0 = direction==0u ? c.Ny : direction==1u ? c.Nz : c.Nx;
	VoxColumn col;
	vox_column(c, direction, a%n0, a/n0, bb, col);
	const bool active = a<A&&!col.out_of_box;
	for(uint32_t base=0u; base<bb.ntri; base+=128u) {
		__syncthreads();
		const uint32_t i = base+threadIdx.x;
		if(i<bb.ntri) {
#pragma unroll
			for(int k=0; k<3; k++) { tri[threadIdx.x][k] = p0[3u*i+k]; tri[threadIdx.x][3+k] = p1[3u*i+k]; tri[threadIdx.x][6+k] = p2[3u*i+k]; }
		}
		__syncthreads();
		if(!active) continue;
		const uint32_t cnt = bb.ntri-base<128u ? bb.ntri-base : 128u;
		for(uint32_t k=0u; k<cnt; k++) vox_cross(col, tri[k][0], tri[k][1], tri[k][2], tri[k][3], tri[k][4], tri[k][5], tri[k][6], tri[k][7], tri[k][8]);
	}
	if(!active) return;
	vox_fill(c, direction, flag, bb, col);
}
// The same with a bin grid over the face (csrc/vox_bins.h): one block per bin of 32 x 4 columns, which walks the bin's triangle list only -- the triangles whose
// projected bounding box, padded by one cell, reaches one of its columns, in ascending triangle order. A ray meets the triangles that can cross it in the order the
// kernel above meets them, so the crossings (and which 64 are kept when there are more) and the flags are the same; the work drops from columns x triangles to
// columns x (triangles near the column). The pad is the reference's own margin for handing a domain only "its" triangles (FX/lbm.cpp:41-90). All threads of a block
// read the same triangle at the same time: one broadcast transaction per warp and load.
__global__ void __launch_bounds__(128) k_voxelize_mesh_binned(const __grid_constant__ DomainConst c, const uint32_t direction, const uint8_t flag, const VoxBox bb, const uint32_t bins0,
	const uint32_t* __restrict__ bin_start, const uint32_t* __restrict__ bin_ids, const float* __restrict__ p0, const float* __restrict__ p1, const float* __restrict__ p2) {
	const uint32_t n0 = direction==0u ? c.Ny : direction==1u ? c.Nz : c.Nx, n1 = direction==0u ? c.Nz : direction==1u ? c.Nx : c.Ny;
	const uint32_t c0 = (blockIdx.x%bins0)*32u+(threadIdx.x&31u), c1 = (blockIdx.x/bins0)*4u+(threadIdx.x>>5);
	if(c0>=n0||c1>=n1) return;
	VoxColumn col;
	vox_column(c, direction, c0, c1, bb, col);
	if(col.out_of_box) return;
	const uint32_t end = __ldg(bin_start+blockIdx.x+1u);
	for(uint32_t k=__ldg(bin_start+blockIdx.x); k<end; k++) {
		const uint32_t i = __ldg(bin_ids+k);
		vox_cross(col, __ldg(p0+3u*i), __ldg(p0+3u*i+1u), __ldg(p0+3u*i+2u), __ldg(p1+3u*i), __ldg(p1+3u*i+1u), __ldg(p1+3u*i+2u), __ldg(p2+3u*i), __ldg(p2+3u*i+1u), __ldg(p2+3u*i+2u));
	}
	vox_fill(c, direction, flag, bb, col);
}

// FAST variant: cos(phase + phi) = cos(phase) cos(phi) - sin(phase) sin(phi). The per-mode products A*cos(phi), A*sin(phi) come from a table built once on
// the host (luw_vk_inlet_create); per point and mode ONE range-reduced hardware sine / cosine pair replaces three library cosines.
// cs[6*V]: Ax cos(phix), Ax sin(phix), Ay cos(phiy), Ay sin(phiy), Az cos(phiz), Az sin(phiz). Absolute error per term ~1e-6 |A|. One difference in kind: the
// reference rounds phase + phi to a float before the cosine (half an ulp of the phase: 1e-4 rad once omega*t reaches thousands of radians), the identity
// does not -- late in a run the two agree to that rounding, not to 1e-6 (tests/test_gpu_parity.py states both tolerances).
__device__ __forceinline__ void sincos_reduced(const float ph, float& s, float& c) {
	const float k = rintf(ph*0.15915494309189535f); // phase / 2 pi
	float r = fmaf(-k, 6.2831854820251465f, ph); // 2 pi split in two floats (Cody-Waite)
	r = fmaf(-k, -1.7484555e-7f, r);
	__sincosf(r, &s, &c);
}
__global__ void __launch_bounds__(128) k_vk_inlet_apply_fast(const uint64_t Ncells, const uint32_t use_interp, const float t0, const float t1, const float alpha,
	const uint64_t P, const uint64_t M, const uint64_t V, const uint64_t* __restrict__ point_cell, const uint8_t* __restrict__ point_face,
	const float* __restrict__ pd, const float* __restrict__ md, const float* __restrict__ cs, float* __restrict__ u) {
	const uint64_t i = (uint64_t)blockIdx.x*blockDim.x+threadIdx.x;
	if(i>=P) return;
	const uint64_t n = point_cell[i];
	const uint64_t fid = point_face[i]&0x07u;
	const float px = pd[i], py = pd[P+i], pz = pd[2ull*P+i];
	const float ubx = pd[3ull*P+i], uby = pd[4ull*P+i], ubz = pd[5ull*P+i], sigma = pd[6ull*P+i];
	if(fid>=5ull||!(sigma>0.0f)) { u[n] = ubx; u[Ncells+n] = uby; u[2ull*Ncells+n] = ubz; return; }
	float qx = 0.0f, qy = 0.0f, qz = 0.0f;
	for(uint64_t m=0ull; m<M; m++) {
		const uint64_t k = fid*M+m;
		const float kx = __ldg(md+k), ky = __ldg(md+V+k), kz = __ldg(md+2ull*V+k), om = __ldg(md+3ull*V+k);
		const float axc = __ldg(cs+k), axs = __ldg(cs+V+k), ayc = __ldg(cs+2ull*V+k), ays = __ldg(cs+3ull*V+k), azc = __ldg(cs+4ull*V+k), azs = __ldg(cs+5ull*V+k);
		float s, c;
		sincos_reduced(fmaf(kx, px, fmaf(ky, py, fmaf(kz, pz, om*t0))), s, c); // the phase is formed exactly like the reference forms it
		float vx = fmaf(c, axc, -s*axs), vy = fmaf(c, ayc, -s*ays), vz = fmaf(c, azc, -s*azs);
		if(use_interp!=0u) {
			sincos_reduced(fmaf(kx, px, fmaf(ky, py, fmaf(kz, pz, om*t1))), s, c);
			const float vx1 = fmaf(c, axc, -s*axs), vy1 = fmaf(c, ayc, -s*ays), vz1 = fmaf(c, azc, -s*azs);
			vx = fmaf(alpha, vx1-vx, vx); vy = fmaf(alpha, vy1-vy, vy); vz = fmaf(alpha, vz1-vz, vz);
		}
		qx += vx; qy += vy; qz += vz;
	}
	u[n] = fmaf(sigma, qx, ubx); u[Ncells+n] = fmaf(sigma, qy, uby); u[2ull*Ncells+n] = fmaf(sigma, qz, ubz);
}

} // anonymous namespace
} // namespace luw
