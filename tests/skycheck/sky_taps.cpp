// sky_taps.cpp — TEST HARNESS (compiled by tests/test_sky_light.py with the host check's flags, never part of libb2r.so).
//
// The product's B2R_FLAG_SKY_LIGHT routines (csrc/b2r_shade.h, csrc/b2r_host.cpp) on the CPU, for the CPU-only test tier. The dielectric taps
// (tests/dielcheck/diel_taps.cpp, unchanged) are included whole, and with them the host check. sk_render_sample is their dc_render_sample with
// the SKY shading routines and a lens: the control flow of one path through k_bounce_brute / k_intersect_closest + k_shade + k_intersect_shadow
// with the sky instantiations, reading the tables of the host twin build_sky_tables.
#include "../dielcheck/diel_taps.cpp"

extern "C" {

// the host twin's tables of a w x h texture: marg[rows + 1], cond[rows][cols + 1], pdf[h][w] (any may be null: sizes only); returns 0
int sk_build_tables(const float* rgba, int32_t w, int32_t h, const float ambient[3], float* marg, float* cond, float* pdf, uint32_t* cols, uint32_t* rows) {
	SkyTables t; build_sky_tables(reinterpret_cast<const float4*>(rgba), w, h, ambient, t);
	*cols = t.cols; *rows = t.rows;
	if (marg) std::memcpy(marg, t.marg.data(), t.marg.size() * sizeof(float));
	if (cond) std::memcpy(cond, t.cond.data(), t.cond.size() * sizeof(float));
	if (pdf) std::memcpy(pdf, t.pdf.data(), t.pdf.size() * sizeof(float));
	return 0;
}
// sky_texels_valid: returns 1 = valid; *nonzero
int sk_texels_valid(const float* rgba, size_t n, const float ambient[3], int* nonzero) {
	bool nz = false; const bool ok = sky_texels_valid(reinterpret_cast<const float4*>(rgba), n, ambient, &nz);
	*nonzero = nz ? 1 : 0; return ok ? 1 : 0;
}
// sky_sample_dir for n draws u[n][4] = {um, uc, uy, ux}: dirs[n][3], cells[n] (texel index of the drawn cell), texels[n] (texel of the lookup)
void sk_sample_dirs(const float* marg, const float* cond, uint32_t cols, uint32_t rows, int32_t w, int32_t h, const float* u, uint32_t n, float* dirs, int32_t* cells, int32_t* texels) {
	SkyDev sky{marg, cond, nullptr, cols, rows, 1.0f, 0.0f};
	SceneDev sc{}; sc.hdri_w = w; sc.hdri_h = h; sc.hdri_fw = static_cast<float>(w - 1); sc.hdri_fh = static_cast<float>(h - 1);
	for (uint32_t k = 0; k < n; k++) {
		const f3 d = sky_sample_dir(sky, w, u[4 * k], u[4 * k + 1], u[4 * k + 2], u[4 * k + 3], cells + k);
		dirs[3 * k] = d.x; dirs[3 * k + 1] = d.y; dirs[3 * k + 2] = d.z;
		texels[k] = sky_texel(sc, d.x, d.y, d.z);
	}
}
// sky_row_z for j = 0..rows
void sk_row_z(uint32_t rows, float* out) { for (uint32_t j = 0; j <= rows; j++) out[j] = sky_row_z(j, rows); }

// One sample (`acc`) for every pixel, as dc_render_sample, with flags B2R_FLAG_SKY_LIGHT (SKY routines, the host twin's tables when the sky is
// sampled), B2R_FLAG_DIELECTRIC, and a lens of radius lens[0] > 0 focused at lens[1] (null: pinhole). counters as dc_render_sample's.
int sk_render_sample(const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_prims, uint32_t n_nodes,
                     const b2r_material* materials, uint32_t n_mat, const int32_t* lights, uint32_t n_lights,
                     const b2r_sphere* geometry, const float cam11[11], uint32_t width, uint32_t height,
                     uint32_t max_bounces, uint32_t flags, uint32_t acc, int use_bvh, float* rad_out, uint64_t counters[5],
                     const float ambient[3], const float* hdri_rgba, int32_t hdri_w, int32_t hdri_h, const float* lens) {
	PackedScene ps; pack_scene(prims, n_prims, materials, n_mat, lights, n_lights, geometry, ps);
	WideBvh wide;
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, cam11, 1);
	if (use_bvh == 2) { std::vector<b2r_bvh_node> tree; build_traversal_tree(prims, n_prims, tree); flatten_bvh(tree.data(), static_cast<uint32_t>(tree.size()), prims, n_prims, wide, &ob); }
	else flatten_bvh(nodes, n_nodes, prims, n_prims, wide, &ob);
	if (wide.max_stack + 3u > static_cast<uint32_t>(kTraversalStack)) return B2R_ERR_BVH;
	std::vector<uint32_t> parent, leaf_node; hc_link_tables(wide, n_prims, parent, leaf_node);
	SceneDev sc{};
	sc.parent = parent.data();
	sc.prims = ps.prims.data(); sc.prim_mat = ps.prim_mat.data(); sc.mat_albedo = ps.mat_albedo.data(); sc.mat_emission = ps.mat_emission.data(); sc.mat_f0 = ps.mat_f0.data();
	sc.light_sphere = ps.light_sphere.data(); sc.light_emit = ps.light_emit.data(); sc.wide = wide.nodes.data(); sc.hdri = nullptr;
	sc.n_prims = n_prims; sc.n_mat = n_mat; sc.n_lights = n_lights; sc.light_sel_pdf = 1.0f / static_cast<float>(n_lights);
	sc.has_ambient = (ambient && hdri_rgba && sel_max(ambient[0], sel_max(ambient[1], ambient[2])) > 0.0f) ? 1 : 0;
	if (sc.has_ambient) {
		sc.hdri = reinterpret_cast<const float4*>(hdri_rgba); sc.ambient[0] = ambient[0]; sc.ambient[1] = ambient[1]; sc.ambient[2] = ambient[2];
		sc.hdri_w = hdri_w; sc.hdri_h = hdri_h; sc.hdri_fw = static_cast<float>(hdri_w - 1); sc.hdri_fh = static_cast<float>(hdri_h - 1);
	}
	// SkyDev as b2r.cu's set_sky_scalars fills it
	SkyTables tab; SkyDev sky{};
	bool nonzero = false;
	if ((flags & B2R_FLAG_SKY_LIGHT) && sc.has_ambient) {
		if (!sky_texels_valid(sc.hdri, static_cast<size_t>(hdri_w) * hdri_h, sc.ambient, &nonzero)) return B2R_ERR_ARG;
		if (nonzero) { build_sky_tables(sc.hdri, hdri_w, hdri_h, sc.ambient, tab); sky.marg = tab.marg.data(); sky.cond = tab.cond.data(); sky.pdf = tab.pdf.data(); sky.cols = tab.cols; sky.rows = tab.rows; }
	}
	sky.p_sky = !nonzero ? 0.0f : n_lights == 0u ? 1.0f : 0.5f;
	sky.light_sel_pdf = n_lights ? (1.0f - sky.p_sky) / static_cast<float>(n_lights) : 0.0f;
	const float4* mat_diel = ps.mat_diel.data();
	FrameDev fr{};
	fr.cam = CameraParams{cam11[0], cam11[1], cam11[2], cam11[3], cam11[4], cam11[5], cam11[6], cam11[7], cam11[8], cam11[9], cam11[10]};
	fr.width = width; fr.height = height; fr.h_tiles = width / 16; fr.npix = width * height; fr.h_tiles_magic = magic_for(fr.h_tiles); fr.npix_magic = magic_for(fr.npix); fr.max_bounces = max_bounces; fr.buckets = 1; fr.flags = flags;
	const LensParams lp{lens ? lens[0] : 0.0f, lens ? lens[1] : 0.0f};
	const bool mis = !(flags & B2R_FLAG_NO_MIS);
	std::memset(rad_out, 0, sizeof(float) * 3 * fr.npix);
	for (int k = 0; k < 5; k++) counters[k] = 0;
	uint32_t cs = 0, cb = 0;
	auto trace_all = [&](auto diel_tag, auto sky_tag) {
	constexpr bool DIEL = decltype(diel_tag)::value, SKY = decltype(sky_tag)::value;
	for (uint32_t t = 0; t < fr.npix; t++) {
		PathState s = lp.radius > 0.0f ? primary_path<true>(fr, fr.cam, acc, 0, t, lp) : primary_path(fr, fr.cam, acc, 0, t);
		const uint32_t seed = pixel_seed(t, max_bounces);
		for (uint32_t bounce = 0; bounce < max_bounces; bounce++) {
			counters[0]++;
			const bool last = bounce + 1 >= max_bounces;
			float best = FLT_MAX; int32_t prim = -1;
			if (use_bvh) traverse_closest<false>(sc.wide, wide.tn_bits, Ray{s.ox, s.oy, s.oz, s.dx, s.dy, s.dz}, &best, &prim, &cs, &cb);
			else for (uint32_t j = 0; j < n_prims; j++) {
				const float4 sp = sc.prims[j]; float d;
				if (sphere_hit_closest(sp.x, sp.y, sp.z, sp.w, s.ox, s.oy, s.oz, s.dx, s.dy, s.dz, &d) && d < best) { best = d; prim = static_cast<int32_t>(j); }
			}
			if (prim < 0) {
				if (sc.has_ambient) rad_add(rad_out, fr.npix, s.pid, shade_sky<SKY>(sc, s, bounce, sky), f3{0.0f, 0.0f, 0.0f}, true, false);
				counters[3]++; break;
			}
			counters[2]++;
			const Surface sf = shade_surface<false, DIEL>(sc, s, best, prim, mat_diel);
			if (last) { rad_zero(rad_out, fr.npix, s.pid); counters[4]++; break; }
			ShadowRay sr; bool want_shadow = mis && shade_light_sample<false, DIEL, SKY>(sc, sf, s, prim, acc, seed, bounce, &sr, sky);
			f3 e{0, 0, 0};
			if (sf.emissive) e = shade_emission<DIEL, SKY>(sc, sf, s, best, bounce, mis, sky);
			if (want_shadow) {
				counters[1]++;
				bool occ = false;
				if (use_bvh) occ = traverse_any<false>(sc.wide, Ray{sr.o.x, sr.o.y, sr.o.z, sr.d.x, sr.d.y, sr.d.z}, sr.tfar, &cs, &cb, sc.parent, 0u);
				else for (uint32_t j = 0; j < n_prims && !occ; j++) {
					const float4 sp = sc.prims[j];
					occ = sphere_hit_any(sp.x, sp.y, sp.z, sp.w, sr.o.x, sr.o.y, sr.o.z, sr.d.x, sr.d.y, sr.d.z, sr.tfar);
				}
				if (occ) want_shadow = false;
			}
			if (want_shadow || sf.emissive) rad_add(rad_out, fr.npix, s.pid, sr.L, e, want_shadow, sf.emissive);
			if (!shade_continue<false, DIEL, SKY>(sf, &s, acc, seed, bounce, sky)) { counters[3]++; break; }
		}
	}
	};
	const bool diel = (flags & B2R_FLAG_DIELECTRIC) != 0, sky_on = (flags & B2R_FLAG_SKY_LIGHT) != 0;
	if (flags & B2R_FLAG_GGX) return B2R_ERR_ARG;
	if (diel) { if (sky_on) trace_all(std::true_type{}, std::true_type{}); else trace_all(std::true_type{}, std::false_type{}); }
	else if (sky_on) trace_all(std::false_type{}, std::true_type{}); else trace_all(std::false_type{}, std::false_type{});
	return 0;
}

}  // extern "C"
