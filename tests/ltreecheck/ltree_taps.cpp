// ltree_taps.cpp — TEST HARNESS (compiled by tests/test_light_tree.py with the host check's flags, never part of libb2r.so).
//
// The product's B2R_FLAG_LIGHT_TREE routines (csrc/b2r_shade.h, csrc/b2r_host.cpp) on the CPU, for the CPU-only test tier. The sky taps
// (tests/skycheck/sky_taps.cpp, unchanged) are included whole, and with them the dielectric taps and the host check. lt_render_sample is their
// sk_render_sample with the LTREE shading routines (and GGX, which the sky taps refuse): the control flow of one path through k_bounce_brute /
// k_intersect_closest + k_shade + k_intersect_shadow with the light-tree instantiations, reading the host builder's tree.
#include "../skycheck/sky_taps.cpp"

namespace {
LightTreeDev tree_dev(const LightTree& t, float sel_scale) { return LightTreeDev{t.nodes.data(), t.light.data(), t.prim_light.data(), sel_scale}; }
}  // namespace

extern "C" {

// light_list_valid: 1 = valid
int lt_list_valid(const b2r_material* materials, const int32_t* lights, uint32_t n_lights, const b2r_sphere* geometry) {
	return light_list_valid(materials, lights, n_lights, geometry) ? 1 : 0;
}
// build_light_tree over lights[n] (b2r_sphere) with mean emissions lum[n] and the BVH-order spheres prims[n_prims] (b2r_sphere). Returns the node
// count; any output may be null (sizes only): nodes[n_nodes][8], light[n][4], prim_light[n_prims], lo / hi[n_nodes][3], *depth
uint32_t lt_build(const b2r_sphere* lights, const float* lum, uint32_t n, const b2r_sphere* prims, uint32_t n_prims,
                  float* nodes, int32_t* light, int32_t* prim_light, float* lo, float* hi, uint32_t* depth) {
	std::vector<float4> p(n_prims); std::vector<int32_t> pm(n_prims);
	for (uint32_t i = 0; i < n_prims; i++) { p[i] = make_float4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq); pm[i] = prims[i].material_ID; }
	LightTree t; build_light_tree(lights, lum, n, p.data(), pm.data(), n_prims, t);
	if (nodes) std::memcpy(nodes, t.nodes.data(), t.nodes.size() * sizeof(float4));
	if (light) std::memcpy(light, t.light.data(), t.light.size() * sizeof(int4));
	if (prim_light) std::memcpy(prim_light, t.prim_light.data(), t.prim_light.size() * sizeof(int32_t));
	if (lo) std::memcpy(lo, t.lo.data(), t.lo.size() * sizeof(float));
	if (hi) std::memcpy(hi, t.hi.data(), t.hi.size() * sizeof(float));
	if (depth) *depth = t.depth;
	return static_cast<uint32_t>(t.nodes.size() / 2u);
}
// light_tree_pick for k = 0..m-1 at P[k][3] with u[k]: picked[k], pdf[k] (the descent's product) and pdf_of[k] (light_tree_pdf of the picked light)
void lt_pick(const float* nodes, const int32_t* light, const float* P, const float* u, uint32_t m, int32_t* picked, float* pdf, float* pdf_of) {
	const LightTreeDev lt{reinterpret_cast<const float4*>(nodes), reinterpret_cast<const int4*>(light), nullptr, 1.0f};
	for (uint32_t k = 0; k < m; k++) {
		const f3 p{P[3 * k], P[3 * k + 1], P[3 * k + 2]};
		picked[k] = static_cast<int32_t>(light_tree_pick(lt, p, u[k], pdf + k));
		pdf_of[k] = light_tree_pdf(lt, p, static_cast<uint32_t>(picked[k]));
	}
}
// light_tree_pdf of every light i < n at P: out[n]
void lt_pdf_all(const float* nodes, const int32_t* light, uint32_t n, const float* P, float* out) {
	const LightTreeDev lt{reinterpret_cast<const float4*>(nodes), reinterpret_cast<const int4*>(light), nullptr, 1.0f};
	for (uint32_t i = 0; i < n; i++) out[i] = light_tree_pdf(lt, f3{P[0], P[1], P[2]}, i);
}
// The two selection pdfs of one direction: the light sample's (sel_scale * the descent's pdf, as shade_light_sample forms it) at P[k] with u[k],
// and the emissive hit's (light_tree_hit_pdf of the picked light's BVH-order sphere, as shade_emission forms it) at the same P. Also the pick.
void lt_sel_pair(const float* nodes, const int32_t* light, const int32_t* prim_light, float sel_scale, const float* P, const float* u, uint32_t m,
                 int32_t* picked, float* sel_sample, float* sel_hit) {
	const LightTreeDev lt{reinterpret_cast<const float4*>(nodes), reinterpret_cast<const int4*>(light), prim_light, sel_scale};
	for (uint32_t k = 0; k < m; k++) {
		const f3 p{P[3 * k], P[3 * k + 1], P[3 * k + 2]};
		float t; picked[k] = static_cast<int32_t>(light_tree_pick(lt, p, u[k], &t)); sel_sample[k] = lt.sel_scale * t;
		sel_hit[k] = light_tree_hit_pdf(lt, p, lt.light[picked[k]].x);
	}
}

// One sample (`acc`) for every pixel, as sk_render_sample, with B2R_FLAG_LIGHT_TREE always on (the host builder's tree; B2R_ERR_ARG when the
// light list breaks the input rule), and B2R_FLAG_GGX, B2R_FLAG_DIELECTRIC, B2R_FLAG_SKY_LIGHT and a lens as flags / lens say.
int lt_render_sample(const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_prims, uint32_t n_nodes,
                     const b2r_material* materials, uint32_t n_mat, const int32_t* lights, uint32_t n_lights,
                     const b2r_sphere* geometry, const float cam11[11], uint32_t width, uint32_t height,
                     uint32_t max_bounces, uint32_t flags, uint32_t acc, int use_bvh, float* rad_out, uint64_t counters[5],
                     const float ambient[3], const float* hdri_rgba, int32_t hdri_w, int32_t hdri_h, const float* lens) {
	if (!light_list_valid(materials, lights, n_lights, geometry)) return B2R_ERR_ARG;
	if ((flags & B2R_FLAG_GGX) && (flags & B2R_FLAG_SKY_LIGHT)) return B2R_ERR_ARG;
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
	// SkyDev and LightTreeDev as b2r.cu's set_sky_scalars fills them
	SkyTables tab; SkyDev sky{};
	bool nonzero = false;
	if ((flags & B2R_FLAG_SKY_LIGHT) && sc.has_ambient) {
		if (!sky_texels_valid(sc.hdri, static_cast<size_t>(hdri_w) * hdri_h, sc.ambient, &nonzero)) return B2R_ERR_ARG;
		if (nonzero) { build_sky_tables(sc.hdri, hdri_w, hdri_h, sc.ambient, tab); sky.marg = tab.marg.data(); sky.cond = tab.cond.data(); sky.pdf = tab.pdf.data(); sky.cols = tab.cols; sky.rows = tab.rows; }
	}
	sky.p_sky = !nonzero ? 0.0f : n_lights == 0u ? 1.0f : 0.5f;
	sky.light_sel_pdf = n_lights ? (1.0f - sky.p_sky) / static_cast<float>(n_lights) : 0.0f;
	std::vector<b2r_sphere> lsph(n_lights); std::vector<float> lum(n_lights);
	for (uint32_t i = 0; i < n_lights; i++) { lsph[i] = geometry[lights[i]]; const float* e = materials[lsph[i].material_ID].emission; lum[i] = ((e[0] + e[1]) + e[2]) / 3.0f; }
	LightTree ltree; build_light_tree(lsph.data(), lum.data(), n_lights, ps.prims.data(), ps.prim_mat.data(), n_prims, ltree);
	const LightTreeDev lt = tree_dev(ltree, n_lights ? 1.0f - sky.p_sky : 0.0f);
	const float4* mat_diel = ps.mat_diel.data();
	FrameDev fr{};
	fr.cam = CameraParams{cam11[0], cam11[1], cam11[2], cam11[3], cam11[4], cam11[5], cam11[6], cam11[7], cam11[8], cam11[9], cam11[10]};
	fr.width = width; fr.height = height; fr.h_tiles = width / 16; fr.npix = width * height; fr.h_tiles_magic = magic_for(fr.h_tiles); fr.npix_magic = magic_for(fr.npix); fr.max_bounces = max_bounces; fr.buckets = 1; fr.flags = flags;
	const LensParams lp{lens ? lens[0] : 0.0f, lens ? lens[1] : 0.0f};
	const bool mis = !(flags & B2R_FLAG_NO_MIS);
	std::memset(rad_out, 0, sizeof(float) * 3 * fr.npix);
	for (int k = 0; k < 5; k++) counters[k] = 0;
	uint32_t cs = 0, cb = 0;
	auto trace_all = [&](auto ggx_tag, auto diel_tag, auto sky_tag) {
	constexpr bool GGX = decltype(ggx_tag)::value, DIEL = decltype(diel_tag)::value, SKY = decltype(sky_tag)::value;
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
			const Surface sf = shade_surface<GGX, DIEL>(sc, s, best, prim, mat_diel);
			if (last) { rad_zero(rad_out, fr.npix, s.pid); counters[4]++; break; }
			ShadowRay sr; bool want_shadow = mis && shade_light_sample<GGX, DIEL, SKY, true>(sc, sf, s, prim, acc, seed, bounce, &sr, sky, lt);
			f3 e{0, 0, 0};
			if (sf.emissive) e = shade_emission<DIEL, SKY, true>(sc, sf, s, best, bounce, mis, sky, lt, prim);
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
			if (!shade_continue<GGX, DIEL, SKY, true>(sf, &s, acc, seed, bounce, sky, lt)) { counters[3]++; break; }
		}
	}
	};
	using T = std::true_type; using F = std::false_type;
	const bool ggx = (flags & B2R_FLAG_GGX) != 0, diel = (flags & B2R_FLAG_DIELECTRIC) != 0, sky_on = (flags & B2R_FLAG_SKY_LIGHT) != 0;
	if (ggx) { if (diel) trace_all(T{}, T{}, F{}); else trace_all(T{}, F{}, F{}); }
	else if (diel) { if (sky_on) trace_all(F{}, T{}, T{}); else trace_all(F{}, T{}, F{}); }
	else if (sky_on) trace_all(F{}, F{}, T{}); else trace_all(F{}, F{}, F{});
	return 0;
}

}  // extern "C"
