// diel_taps.cpp — TEST HARNESS (compiled by tests/test_dielectric.py with the host check's flags, never part of libb2r.so).
//
// The product's B2R_FLAG_DIELECTRIC routines (csrc/b2r_shade.h, csrc/b2r_host.cpp) on the CPU, for the CPU-only test tier. The host check
// (tests/hostcheck/hostcheck.cpp, unchanged) is included whole, so its taps (hc_closest_brute, ...) and helpers are available here too;
// dc_render_sample is its hc_render_sample with the DIELECTRIC shading routines added next to the GGX ones: the control flow of one path
// through k_bounce_brute / k_intersect_closest + k_shade + k_intersect_shadow with the dielectric instantiations.
#include "../hostcheck/hostcheck.cpp"

extern "C" {

// One sample (`acc`) for every pixel: rad_out[3][npix] (tile order). counters: ext rays, shadow rays, hits, term, dropped. use_bvh: 0 brute
// force, 1 flattened reference tree, 2 traversal tree. flags: B2R_FLAG_NO_MIS, B2R_FLAG_GGX, B2R_FLAG_DIELECTRIC.
int dc_render_sample(const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_prims, uint32_t n_nodes,
                     const b2r_material* materials, uint32_t n_mat, const int32_t* lights, uint32_t n_lights,
                     const b2r_sphere* geometry, const float cam11[11], uint32_t width, uint32_t height,
                     uint32_t max_bounces, uint32_t flags, uint32_t acc, int use_bvh, float* rad_out, uint64_t counters[5],
                     const float ambient[3], const float* hdri_rgba, int32_t hdri_w, int32_t hdri_h) {
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
	const float4* mat_diel = ps.mat_diel.data();  // Params::mat_diel on the device
	FrameDev fr{};
	fr.cam = CameraParams{cam11[0], cam11[1], cam11[2], cam11[3], cam11[4], cam11[5], cam11[6], cam11[7], cam11[8], cam11[9], cam11[10]};
	fr.width = width; fr.height = height; fr.h_tiles = width / 16; fr.npix = width * height; fr.h_tiles_magic = magic_for(fr.h_tiles); fr.npix_magic = magic_for(fr.npix); fr.max_bounces = max_bounces; fr.buckets = 1; fr.flags = flags;
	const bool mis = !(flags & B2R_FLAG_NO_MIS);
	std::memset(rad_out, 0, sizeof(float) * 3 * fr.npix);
	for (int k = 0; k < 5; k++) counters[k] = 0;
	uint32_t cs = 0, cb = 0;
	auto trace_all = [&](auto ggx_tag, auto diel_tag) {
	constexpr bool GGX = decltype(ggx_tag)::value, DIEL = decltype(diel_tag)::value;
	for (uint32_t t = 0; t < fr.npix; t++) {
		PathState s = primary_path(fr, fr.cam, acc, 0, t);
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
				if (sc.has_ambient) rad_add(rad_out, fr.npix, s.pid, shade_sky(sc, s), f3{0.0f, 0.0f, 0.0f}, true, false);
				counters[3]++; break;
			}
			counters[2]++;
			const Surface sf = shade_surface<GGX, DIEL>(sc, s, best, prim, mat_diel);
			if (last) { rad_zero(rad_out, fr.npix, s.pid); counters[4]++; break; }
			ShadowRay sr; bool want_shadow = mis && shade_light_sample<GGX, DIEL>(sc, sf, s, prim, acc, seed, bounce, &sr);
			f3 e{0, 0, 0};
			if (sf.emissive) e = shade_emission<DIEL>(sc, sf, s, best, bounce, mis);
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
			if (!shade_continue<GGX, DIEL>(sf, &s, acc, seed, bounce)) { counters[3]++; break; }
		}
	}
	};
	const bool ggx = (flags & B2R_FLAG_GGX) != 0, diel = (flags & B2R_FLAG_DIELECTRIC) != 0;
	if (diel) { if (ggx) trace_all(std::true_type{}, std::true_type{}); else trace_all(std::false_type{}, std::true_type{}); }
	else if (ggx) trace_all(std::true_type{}, std::false_type{}); else trace_all(std::false_type{}, std::false_type{});
	return 0;
}

// dielectric_scatter: out = {dir.xyz, F}; returns 1 for a reflection
int dc_scatter(const float v[3], float r, float u0, float out[4]) {
	f3 d; float F; const bool refl = dielectric_scatter(f3{v[0], v[1], v[2]}, r, u0, &d, &F);
	out[0] = d.x; out[1] = d.y; out[2] = d.z; out[3] = F; return refl ? 1 : 0;
}
// dielectric_materials_valid (what b2r_upload_scene / b2r_refit_scene / b2r_set_flags check under B2R_FLAG_DIELECTRIC): 1 = valid
int dc_materials_valid(const b2r_material* materials, uint32_t n_mat) { return dielectric_materials_valid(materials, n_mat) ? 1 : 0; }

}  // extern "C"
