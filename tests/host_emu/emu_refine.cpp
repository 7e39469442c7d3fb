// emu_refine.cpp -- TEST INFRASTRUCTURE: the host emulation of emu.cpp, plus frames whose tile starts are refined on the
// level-8 grid as beam_start_kernel computes them (csrc/ort_beam.cuh, item 2).  Built on demand by tests/host_emu/
// emu_refine.py into tests/host_emu/_build/; never part of libort_b200.so.
#include "emu.cpp"

extern "C" {

// the time limit of the refinement for a camera at the level emu_beam_level picks (ort::beam_fine_t_limit), 0 = none
float emu_refine_fine_t(const float pos[3], const float rot[9], float fov, int W, int H, int depth, const uint32_t* rcp_tab, int log2n)
{
	const int k = emu_beam_level(pos, rot, fov, W, H, depth, rcp_tab, log2n);
	ort::Camera cam{};
	cam.ox = pos[0]; cam.oy = pos[1]; cam.oz = pos[2];
	for (int i = 0; i < 9; ++i) cam.r[i] = rot[i];
	cam.fov = fov;
	cam.aspect = static_cast<float>(W) / static_cast<float>(H);
	cam.vfx = 2.0F / static_cast<float>(W);
	cam.vfy = 2.0F / static_cast<float>(H);
	return ort::beam_fine_t_limit(ort::beam_tile_radius(cam, ort::rcp_table_rel_error(rcp_tab, log2n)), depth, k);
}

// emu_trace_frame with the beam start of every 8 x 4 tile taken from the level-k grid and, where fine_t > 0, refined on
// the level-8 grid `fine` (walker 13, the product's tiers); tau_out (optional): every pixel's tile start
int emu_refine_trace_frame(const uint32_t* nodes8, size_t n_rows, uint32_t root, int depth, float miss_t, const uint32_t* rcp_tab, int log2n,
                           const float pos[3], const float rot[9], float fov, int W, int H, int y0, int rows, int tile_rows, int tile_step,
                           uint32_t* voxel, uint8_t* face, float* t, uint16_t* npush, unsigned long long* stats_out, int nthreads,
                           const uint8_t* beam_skip, int beam_k, const uint8_t* fine, float fine_t, float* tau_out)
{
	const uint32_t* nodes_m1 = nodes8 - 8;
	const ort::RcpTable rt{rcp_tab, 23 - log2n};
	ort::Camera cam;
	cam.ox = pos[0]; cam.oy = pos[1]; cam.oz = pos[2];
	for (int i = 0; i < 9; ++i) cam.r[i] = rot[i];
	cam.fov = fov;
	cam.aspect = static_cast<float>(W) / static_cast<float>(H);
	cam.vfx = 2.0F / static_cast<float>(W);
	cam.vfy = 2.0F / static_cast<float>(H);
	cam.origin_flags = ort::camera_origin_flags(cam.ox, cam.oy, cam.oz, (1u << (23 - depth)) - 1u);
	const int oflags = static_cast<int>(cam.origin_flags);
	const float min_comp = ort::beam_certify_min_comp(cam, ort::beam_tile_radius(cam, ort::rcp_table_rel_error(rcp_tab, log2n)), ort::rcp_table_sig_bits(rcp_tab, log2n));
	const ort::FrameRows fr{ W, H, y0, rows, tile_rows, tile_step, 0, 0, ort::tile_shift_of(tile_rows) };
	Stats total{};
#pragma omp parallel num_threads(nthreads > 0 ? nthreads : 1)
	{
		Stats st{};
		set_bounds(nodes8, n_rows, rcp_tab, log2n);
#pragma omp for schedule(dynamic, 4)
		for (int r = 0; r < rows; ++r)
			for (int x = 0; x < W; ++x)
			{
				float dx, dy, dz;
				ort::camera_ray(cam, x, ort::frame_row(fr, r), dx, dy, dz);
				const ort::Ray ray = ort::ray_setup_camera(rt, cam.ox, cam.oy, cam.oz, dx, dy, dz, cam.origin_flags);
				const float tau = ort::beam_tile_start(ort::BeamGrid{ beam_skip, beam_k }, cam, x & ~7, ort::frame_row(fr, r & ~3), min_comp, nullptr,
				                                       ort::BeamGrid{ fine, ort::kBeamFineLevel }, fine_t);
				if (tau_out) tau_out[static_cast<size_t>(r) * W + x] = tau;
				ort::Hit h;
				if (__float_as_uint(tau) == ort::kBeamAllMissBits)
				{
					// the kernels' whole-tile MISS; the claim behind it (every ray of the tile is a lean-tier ray) is checked here
					h.voxel = 0; h.face = 6; h.t = miss_t; h.npush = 0;
					++st.beam_tile_misses;
					if (!((oflags & static_cast<int>(ort::kOriginInCube)) && ort::lean_path_ok(ray) && fmaxf(ray.bx, fmaxf(ray.by, ray.bz)) < __uint_as_float(0x7F800000u)))
						++st.beam_cert_wrong;
				}
				else h = npush ? walk<true>(13, nodes_m1, root, depth, miss_t, cam.ox, cam.oy, cam.oz, ray, stats_out ? &st : nullptr, oflags, tau)
				               : walk<false>(13, nodes_m1, root, depth, miss_t, cam.ox, cam.oy, cam.oz, ray, stats_out ? &st : nullptr, oflags, tau);
				++st.rays;
				const size_t i = static_cast<size_t>(r) * W + x;
				voxel[i] = h.voxel;
				face[i] = static_cast<uint8_t>(h.face);
				t[i] = h.t;
				if (npush) npush[i] = static_cast<uint16_t>(h.npush < 65535u ? h.npush : 65535u);
			}
		st.oob_loads = g_emu_bounds.violations;
#pragma omp critical
		merge(&total, st);
	}
	if (stats_out) std::memcpy(stats_out, &total, sizeof(total));
	return total.oob_loads ? 1 : 0;
}

}  // extern "C"
