// TEST INFRASTRUCTURE (see cuda_on_host.hpp): the package's kernel SOURCE, compiled for the host, behind a C interface for ctypes.
// Build: g++ -std=c++17 -O2 -ffp-contract=off -fopenmp -shared -fPIC -w -I/usr/local/cuda/include kernels_on_host.cpp -o libluw_kernels_on_host.so
#include "cuda_on_host.hpp"
#include "../../latticeurbanwind_b200/csrc/lbm_kernels.cuh"
#include "../../latticeurbanwind_b200/csrc/vox_bins.h"
using namespace luw;

// one "launch": grid (ceil(Nx/tx), Ny, Nz) x block tx, as launch_cells() of lbm_launch.inc
template<class K> static void for_cells(const DomainConst& c, K kernel) {
	const unsigned tx = c.Nx>=128u ? 128u : c.Nx>=64u ? 64u : 32u, gx = (c.Nx+tx-1u)/tx;
#pragma omp parallel for collapse(2) schedule(static)
	for(long long z=0; z<(long long)c.Nz; z++) for(long long y=0; y<(long long)c.Ny; y++) {
		emu_blockDim = {tx, 1u, 1u}; emu_gridDim = {gx, c.Ny, c.Nz};
		for(unsigned bx=0u; bx<gx; bx++) for(unsigned t=0u; t<tx; t++) { emu_blockIdx = {bx, (unsigned)y, (unsigned)z}; emu_threadIdx = {t, 0u, 0u}; kernel(); }
	}
}
template<class K> static void for_face(const uint32_t A, K kernel) {
	const unsigned gx = (A+127u)/128u;
#pragma omp parallel for schedule(static)
	for(long long b=0; b<(long long)gx; b++) {
		emu_blockDim = {128u, 1u, 1u}; emu_gridDim = {gx, 1u, 1u};
		for(unsigned t=0u; t<128u; t++) { emu_blockIdx = {(unsigned)b, 0u, 0u}; emu_threadIdx = {t, 0u, 0u}; kernel(); }
	}
}
#define BY_PRECISION(c, CALL) switch((c).precision) { case P_FP32: { constexpr int P = P_FP32; CALL; } break; case P_FP16S: { constexpr int P = P_FP16S; CALL; } break; default: { constexpr int P = P_FP16C; CALL; } break; }
#define BY_FEAT(c, CALL) switch((c).features&15u) { case 6u: { constexpr uint32_t F = 6u; CALL; } break; case 15u: { constexpr uint32_t F = 15u; CALL; } break; case 14u: { constexpr uint32_t F = 14u; CALL; } break; case 5u: { constexpr uint32_t F = 5u; CALL; } break; default: return 1; }

extern "C" {
uint64_t emu_sizeof_domain_const() { return sizeof(DomainConst); }
// the strip order of an overlapped halo exchange (csrc/lbm_common.cuh strip_order_fill / strip_of): out[0..4] = so_ylo, so_yhi, so_zlo, so_zhi, so_nb; order[i] = strip id of the i-th strip handed out
int emu_strip_order(uint32_t Ny, uint32_t Nz, uint32_t Dy, uint32_t Dz, uint32_t TY, uint32_t TZ, uint32_t* out, uint32_t* order) {
	DomainConst c; memset(&c, 0, sizeof(c));
	c.Ny = Ny; c.Nz = Nz; c.Dy = Dy; c.Dz = Dz;
	const bool ok = strip_order_fill(c, TY, TZ);
	out[0] = c.so_ylo; out[1] = c.so_yhi; out[2] = c.so_zlo; out[3] = c.so_zhi; out[4] = c.so_nb;
	const uint32_t Ty = (Ny+TY-1u)/TY, Tz = (Nz+TZ-1u)/TZ;
	for(uint32_t i=0u; i<Ty*Tz; i++) order[i] = strip_of(c, i, Ty, Tz);
	return ok ? 1 : 0;
}
// the caller fills a DomainConst through this (same derivations as luw_domain_create) so that the struct layout stays private to C++
int emu_make_domain(DomainConst* c, uint32_t Nx, uint32_t Ny, uint32_t Nz, uint32_t Dx, uint32_t Dy, uint32_t Dz, int Ox, int Oy, int Oz, int precision, uint32_t features, float w,
	int downstream_face, uint32_t buffer_N, float buffer_inv_tau, int nudge_vertical, uint32_t sponge_N, const float* wbuf, const float* sigma,
	void* fi, float* rho, float* u, uint8_t* flags, void* gi, float* T, float w_T, float beta, float T_avg) {
	memset(c, 0, sizeof(*c));
	c->Nx = Nx; c->Ny = Ny; c->Nz = Nz; c->Px = (Nx+15u)&~15u; c->N = (uint64_t)c->Px*Ny*Nz;
	c->Dx = Dx; c->Dy = Dy; c->Dz = Dz; c->Ox = Ox; c->Oy = Oy; c->Oz = Oz;
	c->Nxg = (Nx-2u*(Dx>1u))*Dx; c->Nyg = (Ny-2u*(Dy>1u))*Dy; c->Nzg = (Nz-2u*(Dz>1u))*Dz;
	c->wx = -Ox; c->ex = (int)c->Nxg-1-Ox; c->sy = -Oy; c->ny = (int)c->Nyg-1-Oy; c->tz = (int)c->Nzg-1-Oz;
	c->has_w = c->wx>=0&&c->wx<(int)Nx; c->has_e = c->ex>=0&&c->ex<(int)Nx; c->has_s = c->sy>=0&&c->sy<(int)Ny; c->has_n = c->ny>=0&&c->ny<(int)Ny; c->has_t = c->tz>=0&&c->tz<(int)Nz;
	c->w = w; c->tau0 = 1.0f/w; c->tau0sq = c->tau0*c->tau0; c->precision = precision; c->features = features;
	c->downstream_face = downstream_face; c->buffer_N = buffer_N; c->buffer_inv_tau = buffer_inv_tau; c->nudge_vertical = nudge_vertical; c->sponge_N = sponge_N;
	c->wbuf = wbuf; c->sigma = sigma; c->fi = fi; c->rho = rho; c->u = u; c->flags = flags; c->gi = gi; c->T = T; c->w_T = w_T; c->beta = beta; c->T_avg = T_avg;
	return 0;
}
// the two relaxation-zone tables exactly as luw_domain_create builds them (csrc/luw_cabi.cu: "distance -> sin^2 ramp", "depth -> inv_tau*sin^2 ramp")
void emu_zone_tables(uint32_t buffer_N, uint32_t sponge_N, float sponge_inv_tau, float* wbuf, float* sigma) {
	for(uint32_t k=0u; k<=buffer_N; k++) { const float xi = 1.0f-(float)k/(float)buffer_N; float wb = sinf(1.5707963267948966f*xi); wb *= wb; wbuf[k] = wb; }
	const int Ns = (int)sponge_N;
	for(int k=0; k<Ns; k++) { const float xi = Ns>1 ? 1.0f-(float)k/(float)(Ns-1) : 1.0f; float sg = sinf(1.5707963267948966f*xi); sg = sponge_inv_tau*sg*sg; sigma[k] = sg; }
}
int emu_initialize(const DomainConst* c) { BY_PRECISION(*c, for_cells(*c, [&]{ k_initialize<P>(*c); })); return 0; }
int emu_stream_collide(const DomainConst* c, const StepArgs* a) { BY_PRECISION(*c, BY_FEAT(*c, for_cells(*c, [&]{ k_stream_collide<P, F>(*c, *a); }))); return 0; }
int emu_initialize_thermal(const DomainConst* c) { BY_PRECISION(*c, for_cells(*c, [&]{ k_initialize_thermal<P>(*c); })); return 0; }
int emu_stream_collide_thermal(const DomainConst* c, const StepArgs* a) { BY_PRECISION(*c, BY_FEAT(*c, for_cells(*c, [&]{ k_stream_collide_thermal<P, F>(*c, *a); }))); return 0; }
int emu_update_fields_thermal(const DomainConst* c, const StepArgs* a) {
	if((c->features&6u)!=6u) return 1;
	BY_PRECISION(*c, for_cells(*c, [&]{ k_update_fields_thermal<P, 6u>(*c, *a); }));
	return 0;
}
int emu_halo_gi(const DomainConst* c, uint32_t axis, uint32_t odd, int insert, int xfast, void* bp, void* bm) {
	const uint32_t A = axis==0u ? c->Ny*c->Nz : axis==1u ? c->Nz*c->Nx : c->Nx*c->Ny;
	if(c->precision==P_FP32) { if(insert) for_face(A, [&]{ k_halo_gi<float, true>(*c, axis, A, odd, xfast!=0, (float*)bp, (float*)bm); }); else for_face(A, [&]{ k_halo_gi<float, false>(*c, axis, A, odd, xfast!=0, (float*)bp, (float*)bm); }); }
	else { if(insert) for_face(A, [&]{ k_halo_gi<uint16_t, true>(*c, axis, A, odd, xfast!=0, (uint16_t*)bp, (uint16_t*)bm); }); else for_face(A, [&]{ k_halo_gi<uint16_t, false>(*c, axis, A, odd, xfast!=0, (uint16_t*)bp, (uint16_t*)bm); }); }
	return 0;
}
// the binned voxeliser as luw_voxelize_mesh runs it: bin grid from vox_build_bins, one 128-thread block per bin. stats[0..2] = bins, list entries, longest list
int emu_voxelize_binned(const DomainConst* c, uint32_t direction, uint8_t flag, const float* p0, const float* p1, const float* p2, uint32_t ntri, const float* bbu, uint64_t* stats) {
	const VoxBins bins = vox_build_bins(direction, c->Nx, c->Ny, c->Nz, c->Ox, c->Oy, c->Oz, p0, p1, p2, ntri);
	if(bins.bins0==0u) return 1;
	const VoxBox bb = { ntri, bbu[1], bbu[2], bbu[3], bbu[4], bbu[5], bbu[6] };
	const unsigned nb = bins.bins0*bins.bins1;
	if(stats) { stats[0] = nb; stats[1] = bins.ids.size(); stats[2] = 0ull; for(unsigned b=0u; b<nb; b++) if(bins.start[b+1u]-bins.start[b]>stats[2]) stats[2] = bins.start[b+1u]-bins.start[b]; }
#pragma omp parallel for schedule(dynamic)
	for(long long b=0; b<(long long)nb; b++) {
		emu_blockDim = {128u, 1u, 1u}; emu_gridDim = {nb, 1u, 1u};
		for(unsigned t=0u; t<128u; t++) { emu_blockIdx = {(unsigned)b, 0u, 0u}; emu_threadIdx = {t, 0u, 0u}; k_voxelize_mesh_binned(*c, direction, flag, bb, bins.bins0, bins.start.data(), bins.ids.data(), p0, p1, p2); }
	}
	return 0;
}
int emu_halo_T(const DomainConst* c, uint32_t axis, int insert, int xfast, float* bp, float* bm) {
	const uint32_t A = axis==0u ? c->Ny*c->Nz : axis==1u ? c->Nz*c->Nx : c->Nx*c->Ny;
	if(insert) for_face(A, [&]{ k_halo_T<true>(*c, axis, A, xfast!=0, bp, bm); }); else for_face(A, [&]{ k_halo_T<false>(*c, axis, A, xfast!=0, bp, bm); });
	return 0;
}
}
