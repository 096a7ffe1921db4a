// Command-line driver over the C++ host layer, used by the parity tests (tests/test_cpp_host.py): it does what a case driver does with the
// reference's API (FX/setup.cpp:4931-6153 in miniature): construct LBM, write lbm.flags / lbm.rho / lbm.u through the global accessors,
// set_coriolis, run(steps), read_from_device, and dump rho / u.
//   luw_host_case Nx Ny Nz Dx Dy Dz precision features arith nu steps downstream bufN buf_inv_tau buf_vertical spongeN sponge_inv_tau fx fy fz ox oy oz in.bin out.bin
//   in.bin : flags[N] u8, rho[N] f32, u[3N] f32 (global images, n = x+(y+z*Ny)*Nx);  out.bin : rho[N] f32, u[3N] f32
//   LUW_CASE_TRIANGLES=<file> (u32 n, pmin[3], pmax[3], p0[3n], p1[3n], p2[3n] f32, lattice coordinates): the geometry is voxelised on the device first, through
//   LBM::voxelize_triangles_on_device like FX/setup.cpp:4084-4125 does with the STL, the flags of in.bin are OR-ed on top, and out.bin ends with flags[N] u8
//   LUW_CASE_WIND=h0,h1,... (heights in cells) with LUW_CASE_WIND_THR=t0,t1,... and LUW_CASE_WIND_OUT=<file>: LBM_WindStatistics over the same sampling window as
//   LUW_CASE_STATS; the file gets samples u64, mean_u[3M], comoment[6M], mean_speed[M], m2_speed[M], max_speed[M] f32, exceed[T*M] u32, valid[M] u8, ground[Nx*Ny] u32
//   LUW_CASE_WALL_OUT=<file> (with LUW_CASE_WALL_GROUND=<ground_z>, default 0): LBM_WallLoads over the same sampling window as LUW_CASE_STATS; the file gets
//   samples u64, L u32, K u64, series[samples*L*6] f64, ref_points[3L] f64, column_labels[Nx*Ny] u32, cell[K] u64, label[K] u32, mean_F[3K], m2_F[3K] f32
//   LUW_CASE_PROBES=x0,y0,z0,x1,y1,z1,... (global lattice points) with LUW_CASE_PROBES_OUT=<file>: LBM_Probes sampled after every step of the same window as
//   LUW_CASE_STATS (capacity LUW_CASE_PROBES_CAP, default 256); the file gets samples u64, comps u32, P u64, t[samples] u64, values[samples*comps*P] f32
//   LUW_CASE_PARTICLES=cx,cy,cz,hx,hy,hz,... (box emitters, lattice coordinates) with LUW_CASE_PARTICLES_ARGS=capacity,per_emitter,periodic_mask,wall_mode,seed,
//   bx,by,bz,dt,sigma and LUW_CASE_PARTICLES_OUT=<file>: LBM_Particles over the same window as LUW_CASE_STATS, after every step emit(per_emitter), advance(dt, sigma),
//   count(); the file gets capacity u64, xyz[3*capacity] f64, state[capacity] u8, emitter[capacity] u32, release_t[capacity] u64, samples u64, bins[Bz*By*Bx] u32
//   with LUW_TEMPERATURE in `features`: in.bin carries T[N] f32 after u, out.bin ends with T[N] f32; alpha / beta of the LBM constructor from LUW_CASE_ALPHA / LUW_CASE_BETA
#include "lbm.hpp"
#include <fstream>
#include <sstream>

template<typename T> static std::vector<T> env_list(const char* name) { // comma-separated numbers, empty if unset
	std::vector<T> v;
	const char* e = getenv(name);
	if(!e) return v;
	std::stringstream ss(e);
	std::string item;
	while(std::getline(ss, item, ',')) if(!item.empty()) v.push_back((T)atof(item.c_str()));
	return v;
}

int main(int argc, char** argv) {
	if(argc!=26) { fprintf(stderr, "usage: see host_case.cpp\n"); return 2; }
	int a = 1;
	const uint Nx = (uint)atoi(argv[a++]), Ny = (uint)atoi(argv[a++]), Nz = (uint)atoi(argv[a++]);
	const uint Dx = (uint)atoi(argv[a++]), Dy = (uint)atoi(argv[a++]), Dz = (uint)atoi(argv[a++]);
	lbm_settings.precision = (uint)atoi(argv[a++]);
	lbm_settings.features = (uint)atoi(argv[a++])&~(uint)(LUW_BUFFER_NUDGING|LUW_TOP_SPONGE);
	const uint want = (uint)atoi(argv[a-1]);
	lbm_settings.arith = (uint)atoi(argv[a++]);
	const float nu = (float)atof(argv[a++]);
	const ulong steps = (ulong)atoll(argv[a++]);
	lbm_settings.downstream_face = atoi(argv[a++]);
	const uint bufN = (uint)atoi(argv[a++]); const float buf_inv_tau = (float)atof(argv[a++]); const bool buf_vertical = atoi(argv[a++])!=0;
	const uint spongeN = (uint)atoi(argv[a++]); const float sponge_inv_tau = (float)atof(argv[a++]);
	if(want&LUW_BUFFER_NUDGING) lbm_settings.set_buffer_nudging(bufN, buf_inv_tau, buf_vertical);
	if(want&LUW_TOP_SPONGE) lbm_settings.set_top_sponge(spongeN, sponge_inv_tau);
	const float fx = (float)atof(argv[a++]), fy = (float)atof(argv[a++]), fz = (float)atof(argv[a++]);
	const float ox = (float)atof(argv[a++]), oy = (float)atof(argv[a++]), oz = (float)atof(argv[a++]);
	const char* in_path = argv[a++]; const char* out_path = argv[a++];

	const bool thermal = (want&LUW_TEMPERATURE)!=0u;
	const float alpha = thermal&&getenv("LUW_CASE_ALPHA") ? (float)atof(getenv("LUW_CASE_ALPHA")) : 0.0f, beta = thermal&&getenv("LUW_CASE_BETA") ? (float)atof(getenv("LUW_CASE_BETA")) : 0.0f;
	LBM lbm(uint3(Nx, Ny, Nz), Dx, Dy, Dz, nu, fx, fy, fz, 0.0f, alpha, beta);
	lbm.set_coriolis(ox, oy, oz);
	const ulong N = lbm.get_N();
	std::vector<uchar> flags(N); std::vector<float> rho(N), u(3ull*N);
	std::ifstream in(in_path, std::ios::binary);
	in.read((char*)flags.data(), (std::streamsize)N); in.read((char*)rho.data(), (std::streamsize)(4ull*N)); in.read((char*)u.data(), (std::streamsize)(12ull*N));
	std::vector<float> T(thermal ? N : 0ull);
	if(thermal) in.read((char*)T.data(), (std::streamsize)(4ull*N));
	if(!in) print_error("cannot read the input images");
	if(thermal) for(ulong n=0ull; n<N; n++) lbm.T[n] = T[n]; // FX/setup.cpp:5268-5317 writes lbm.T the same way
	const char* tri_path = getenv("LUW_CASE_TRIANGLES");
	if(tri_path) {
		std::ifstream tf(tri_path, std::ios::binary);
		uint ntri = 0u; float bb[6];
		tf.read((char*)&ntri, 4); tf.read((char*)bb, 24);
		std::vector<float> p0(3ull*ntri), p1(3ull*ntri), p2(3ull*ntri);
		tf.read((char*)p0.data(), (std::streamsize)(12ull*ntri)); tf.read((char*)p1.data(), (std::streamsize)(12ull*ntri)); tf.read((char*)p2.data(), (std::streamsize)(12ull*ntri));
		if(!tf) print_error("cannot read the triangle file");
		const std::vector<uint> given = lbm.voxelize_triangles_on_device(p0.data(), p1.data(), p2.data(), ntri, float3(bb[0], bb[1], bb[2]), float3(bb[3], bb[4], bb[5]));
		for(uint d=0u; d<lbm.get_D(); d++) printf("luw_host_case: domain %u voxelised %u of %u triangles\n", d, given[d], ntri);
		lbm.flags.read_from_device(); // host mirrors of all domains, like FX/lbm.cpp:1641-1644
	}
	for(ulong n=0ull; n<N; n++) { // the way FX/setup.cpp writes boundary conditions: through the stitched global accessors
		lbm.flags[n] = tri_path ? (uchar)(lbm.flags[n]|flags[n]) : flags[n]; lbm.rho[n] = rho[n];
		lbm.u.x[n] = u[n]; lbm.u.y[n] = u[N+n]; lbm.u.z[n] = u[2ull*N+n];
	}
	lbm.run(0ull); // initialise only (FX/setup.cpp:4852)
	const ulong samples = getenv("LUW_CASE_STATS") ? (ulong)atoll(getenv("LUW_CASE_STATS")) : 0ull; // averaging window over the last `samples` steps (FX/setup.cpp:4510-4542)
	LBM_Statistics* stats = samples>0ull ? new LBM_Statistics(lbm) : nullptr;
	const char* wind_out = getenv("LUW_CASE_WIND_OUT");
	LBM_WindStatistics* wind = wind_out ? new LBM_WindStatistics(lbm, env_list<uint>("LUW_CASE_WIND"), env_list<float>("LUW_CASE_WIND_THR")) : nullptr;
	lbm.run(steps-(samples<steps ? samples : steps));
	const char* wall_out = getenv("LUW_CASE_WALL_OUT");
	LBM_WallLoads* wall = wall_out ? new LBM_WallLoads(lbm, getenv("LUW_CASE_WALL_GROUND") ? (uint)atoi(getenv("LUW_CASE_WALL_GROUND")) : 0u) : nullptr;
	const char* probes_out = getenv("LUW_CASE_PROBES_OUT");
	LBM_Probes* probes = probes_out ? new LBM_Probes(lbm, env_list<uint>("LUW_CASE_PROBES"), getenv("LUW_CASE_PROBES_CAP") ? (uint)atoi(getenv("LUW_CASE_PROBES_CAP")) : 256u) : nullptr;
	const char* particles_out = getenv("LUW_CASE_PARTICLES_OUT");
	const std::vector<double> pargs = env_list<double>("LUW_CASE_PARTICLES_ARGS");
	if(particles_out&&pargs.size()!=10u) print_error("LUW_CASE_PARTICLES_ARGS needs 10 values");
	LBM_Particles* particles = particles_out ? new LBM_Particles(lbm, env_list<double>("LUW_CASE_PARTICLES"), (ulong)pargs[0], (uint)pargs[2], (uint)pargs[3], (ulong)pargs[4],
		(uint)pargs[5], (uint)pargs[6], (uint)pargs[7]) : nullptr;
	for(ulong k=0ull; k<(samples<steps ? samples : steps); k++) {
		lbm.run(1ull);
		if(probes) probes->sample();
		if(particles) { particles->emit((uint)pargs[1]); particles->advance((float)pargs[8], pargs[9]); particles->count(); }
		stats->accumulate(); if(wind) wind->accumulate(); if(wall) wall->accumulate();
	}
	if(particles) {
		std::vector<double> xyz; std::vector<uchar> state; std::vector<uint> emitter, bins; std::vector<ulong> release_t;
		particles->download(xyz, state, emitter, release_t);
		const uint64_t count = (uint64_t)particles->download_bins(bins), K = (uint64_t)particles->capacity;
		std::ofstream pf(particles_out, std::ios::binary);
		pf.write((const char*)&K, 8); pf.write((const char*)xyz.data(), (std::streamsize)(8u*xyz.size())); pf.write((const char*)state.data(), (std::streamsize)state.size());
		pf.write((const char*)emitter.data(), (std::streamsize)(4u*emitter.size())); pf.write((const char*)release_t.data(), (std::streamsize)(8u*release_t.size()));
		pf.write((const char*)&count, 8); pf.write((const char*)bins.data(), (std::streamsize)(4u*bins.size()));
		delete particles;
	}
	if(probes) {
		std::vector<float> values;
		const uint64_t count = (uint64_t)probes->series(values), P = (uint64_t)probes->points;
		std::ofstream pf(probes_out, std::ios::binary);
		pf.write((const char*)&count, 8); pf.write((const char*)&probes->comps, 4); pf.write((const char*)&P, 8);
		pf.write((const char*)probes->t.data(), (std::streamsize)(8u*probes->t.size())); pf.write((const char*)values.data(), (std::streamsize)(4u*values.size()));
		delete probes;
	}
	if(wall) {
		std::vector<double> series; std::vector<ulong> cell; std::vector<uint> label; std::vector<float> mean_F, m2_F;
		const uint64_t count = (uint64_t)wall->series(series), K = (uint64_t)(wall->surface(cell, label, mean_F, m2_F), cell.size());
		std::ofstream wf(wall_out, std::ios::binary);
		wf.write((const char*)&count, 8); wf.write((const char*)&wall->L, 4); wf.write((const char*)&K, 8);
		wf.write((const char*)series.data(), (std::streamsize)(8u*series.size())); wf.write((const char*)wall->ref_points.data(), (std::streamsize)(8u*wall->ref_points.size()));
		wf.write((const char*)wall->column_labels.data(), (std::streamsize)(4u*wall->column_labels.size()));
		wf.write((const char*)cell.data(), (std::streamsize)(8u*K)); wf.write((const char*)label.data(), (std::streamsize)(4u*K));
		wf.write((const char*)mean_F.data(), (std::streamsize)(4u*mean_F.size())); wf.write((const char*)m2_F.data(), (std::streamsize)(4u*m2_F.size()));
		delete wall;
	}
	if(wind) {
		std::vector<float> mean_u, comoment, mean_speed, m2_speed, max_speed; std::vector<uint> exceed; std::vector<uchar> valid;
		const uint64_t count = (uint64_t)wind->download(mean_u, comoment, mean_speed, m2_speed, max_speed, exceed, valid);
		std::ofstream wf(wind_out, std::ios::binary);
		wf.write((const char*)&count, 8);
		for(const std::vector<float>* v : { &mean_u, &comoment, &mean_speed, &m2_speed, &max_speed }) wf.write((const char*)v->data(), (std::streamsize)(4u*v->size()));
		wf.write((const char*)exceed.data(), (std::streamsize)(4u*exceed.size())); wf.write((const char*)valid.data(), (std::streamsize)valid.size());
		wf.write((const char*)wind->ground.data(), (std::streamsize)(4u*wind->ground.size()));
		delete wind;
	}
	lbm.rho.read_from_device(); lbm.u.read_from_device();
	for(ulong n=0ull; n<N; n++) { rho[n] = lbm.rho[n]; u[n] = lbm.u.x[n]; u[N+n] = lbm.u.y[n]; u[2ull*N+n] = lbm.u.z[n]; }
	std::ofstream out(out_path, std::ios::binary);
	out.write((const char*)rho.data(), (std::streamsize)(4ull*N)); out.write((const char*)u.data(), (std::streamsize)(12ull*N));
	if(samples>0ull) { // avg_u[3N] interleaved, avg_rho[N], M2_u[N], M2_v[N], M2_w[N]
		std::vector<float> avg_u, avg_rho, M2_u, M2_v, M2_w;
		const ulong count = stats->download(avg_u, avg_rho, M2_u, M2_v, M2_w);
		if(count!=(samples<steps ? samples : steps)) print_error("statistics sample count is off");
		out.write((const char*)avg_u.data(), (std::streamsize)(12ull*N)); out.write((const char*)avg_rho.data(), (std::streamsize)(4ull*N));
		out.write((const char*)M2_u.data(), (std::streamsize)(4ull*N)); out.write((const char*)M2_v.data(), (std::streamsize)(4ull*N)); out.write((const char*)M2_w.data(), (std::streamsize)(4ull*N));
	}
	if(thermal) {
		lbm.T.read_from_device();
		for(ulong n=0ull; n<N; n++) T[n] = lbm.T[n];
		out.write((const char*)T.data(), (std::streamsize)(4ull*N));
	}
	if(tri_path) {
		lbm.flags.read_from_device();
		for(ulong n=0ull; n<N; n++) flags[n] = lbm.flags[n];
		out.write((const char*)flags.data(), (std::streamsize)N);
	}
	delete stats;
	printf("luw_host_case: %llu cells, %u domain(s), %llu steps, t = %llu\n", (unsigned long long)N, lbm.get_D(), (unsigned long long)steps, (unsigned long long)lbm.get_t());
	return 0;
}
