// hostcheck.cpp — TEST HARNESS (built by tests/conftest.py with g++, never part of libb2r.so).
//
// Runs the product's own host+device routines (csrc/b2r_math.h, csrc/b2r_shade.h, csrc/b2r_host.cpp) on the CPU so the
// CPU-only test tier can compare them bit-for-bit with the oracle on the build box, where no GPU exists. The control
// flow below mirrors one path through k_bounce_brute / k_intersect_closest + k_shade + k_intersect_shadow
// (csrc/b2r_device.cuh); the GPU tier (-m gpu) then checks the kernels themselves through the C ABI.
#include "b2r_shade.h"
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

using namespace b2r;

// Host twin of the GPU refit (k_refit_level runs the same shared routine, refit_slot in csrc/b2r_shade.h, one thread per slot and one
// launch per level): levels deepest first, children always sit on a deeper level. Lives in the test harness — libb2r refits on the GPU only.
static void refit_wide(WideBvh& tree, const float4* prims, const uint32_t* remap, const OriginBox& ob) {
	float4* wide = reinterpret_cast<float4*>(tree.nodes.data());
	for (size_t l = tree.level_first.size() - 1; l-- > 0;)
		for (uint32_t i = tree.level_first[l]; i < tree.level_first[l + 1]; i++) for (int k = 0; k < 4; k++) refit_slot(wide, prims, remap, ob, i, k);
	tree.cost = wide_cost(tree);
}
// the origin box of a test: `box6` ({lo.xyz, hi.xyz}, e.g. b2r_get_origin_box of the context under test) when given, else the library's
// rule over the spheres plus the given points (camera position, ray origins)
static OriginBox origin_box_of(const b2r_sphere* prims, uint32_t n, const float* box6, const float* points, uint32_t n_points) {
	if (box6) { OriginBox ob; for (int k = 0; k < 3; k++) { ob.lo[k] = box6[k]; ob.hi[k] = box6[3 + k]; } return ob; }
	float lo[3], hi[3]; sphere_bounds(prims, n, lo, hi);
	return origin_box_rule(lo, hi, points, n_points);
}
static void ray_origin_bounds(const float* rays, uint32_t n, float out[6]) {
	for (int k = 0; k < 3; k++) { out[k] = FLT_MAX; out[3 + k] = -FLT_MAX; }
	for (uint32_t i = 0; i < n; i++) for (int k = 0; k < 3; k++) { out[k] = fminf(out[k], rays[6 * static_cast<size_t>(i) + k]); out[3 + k] = fmaxf(out[3 + k], rays[6 * static_cast<size_t>(i) + k]); }
}

// the tables k_link_tables writes: the wide node that links to node i (the root's entry is 0) and the node holding sphere i's leaf slot
static void hc_link_tables(const WideBvh& w, uint32_t n_prims, std::vector<uint32_t>& parent, std::vector<uint32_t>& leaf_node) {
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	const uint32_t nn = static_cast<uint32_t>(w.nodes.size());
	parent.assign(nn, 0u); leaf_node.assign(n_prims, 0u);
	for (uint32_t nd = 0; nd < nn; nd++) for (int k = 0; k < 4; k++) {
		const int32_t l = as_int(wide[static_cast<size_t>(nd) * 8 + 2 * k + 1].z);
		if (l == kEmptyLink) continue;
		if (l < 0) leaf_node[~l] = nd; else parent[l] = nd;
	}
}

extern "C" {

// One sample (`acc`) for every pixel: rad_out[3][npix] (tile order). counters: ext rays, shadow rays, hits, term, dropped.
// use_bvh: 0 brute force, 1 flattened reference tree, 2 traversal tree (libb2r's default).
int hc_render_sample(const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_prims, uint32_t n_nodes,
                     const b2r_material* materials, uint32_t n_mat, const int32_t* lights, uint32_t n_lights,
                     const b2r_sphere* geometry, const float cam11[11], uint32_t width, uint32_t height,
                     uint32_t max_bounces, uint32_t flags, uint32_t acc, int use_bvh, float* rad_out, uint64_t counters[5],
                     const float ambient[3], const float* hdri_rgba, int32_t hdri_w, int32_t hdri_h) {  // sky (Primitives.hpp:29-47): hdri may be null when ambient is 0
	PackedScene ps; pack_scene(prims, n_prims, materials, n_mat, lights, n_lights, geometry, ps);
	WideBvh wide;
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, cam11, 1);  // spheres + camera position
	if (use_bvh == 2) { std::vector<b2r_bvh_node> tree; build_traversal_tree(prims, n_prims, tree); flatten_bvh(tree.data(), static_cast<uint32_t>(tree.size()), prims, n_prims, wide, &ob); }  // what libb2r uploads by default
	else flatten_bvh(nodes, n_nodes, prims, n_prims, wide, &ob);  // B2R_FLAG_REFERENCE_TREE
	if (wide.max_stack + 3u > static_cast<uint32_t>(kTraversalStack)) return B2R_ERR_BVH;
	std::vector<uint32_t> parent, leaf_node; hc_link_tables(wide, n_prims, parent, leaf_node);
	SceneDev sc{};
	sc.parent = parent.data();
	sc.prims = ps.prims.data(); sc.prim_mat = ps.prim_mat.data(); sc.mat_albedo = ps.mat_albedo.data(); sc.mat_emission = ps.mat_emission.data(); sc.mat_f0 = ps.mat_f0.data();
	sc.light_sphere = ps.light_sphere.data(); sc.light_emit = ps.light_emit.data(); sc.wide = wide.nodes.data(); sc.hdri = nullptr;
	sc.n_prims = n_prims; sc.n_mat = n_mat; sc.n_lights = n_lights; sc.light_sel_pdf = 1.0f / static_cast<float>(n_lights);
	sc.has_ambient = (ambient && hdri_rgba && sel_max(ambient[0], sel_max(ambient[1], ambient[2])) > 0.0f) ? 1 : 0;  // Renderer.hpp:79
	if (sc.has_ambient) {
		sc.hdri = reinterpret_cast<const float4*>(hdri_rgba); sc.ambient[0] = ambient[0]; sc.ambient[1] = ambient[1]; sc.ambient[2] = ambient[2];
		sc.hdri_w = hdri_w; sc.hdri_h = hdri_h; sc.hdri_fw = static_cast<float>(hdri_w - 1); sc.hdri_fh = static_cast<float>(hdri_h - 1);  // Application.cpp:230-231
	}
	FrameDev fr{};
	fr.cam = CameraParams{cam11[0], cam11[1], cam11[2], cam11[3], cam11[4], cam11[5], cam11[6], cam11[7], cam11[8], cam11[9], cam11[10]};
	fr.width = width; fr.height = height; fr.h_tiles = width / 16; fr.npix = width * height; fr.h_tiles_magic = magic_for(fr.h_tiles); fr.npix_magic = magic_for(fr.npix); fr.max_bounces = max_bounces; fr.buckets = 1; fr.flags = flags;
	const bool mis = !(flags & B2R_FLAG_NO_MIS);
	std::memset(rad_out, 0, sizeof(float) * 3 * fr.npix);
	for (int k = 0; k < 5; k++) counters[k] = 0;
	uint32_t cs = 0, cb = 0;
	auto trace_all = [&](auto ggx_tag) {  // B2R_FLAG_GGX: the same loop with the GGX closure's shading routines (k_shade<EXACT, GGX> / k_bounce_brute<..., GGX>)
	constexpr bool GGX = decltype(ggx_tag)::value;
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
			if (prim < 0) {  // miss: terminated; with an ambient sky the miss shader adds its texel (Renderer.hpp:411-420), as the kernels do
				if (sc.has_ambient) rad_add(rad_out, fr.npix, s.pid, shade_sky(sc, s), f3{0.0f, 0.0f, 0.0f}, true, false);
				counters[3]++; break;
			}
			counters[2]++;
			const Surface sf = shade_surface<GGX>(sc, s, best, prim);
			if (last) { rad_zero(rad_out, fr.npix, s.pid); counters[4]++; break; }
			ShadowRay sr; bool want_shadow = mis && shade_light_sample<GGX>(sc, sf, s, prim, acc, seed, bounce, &sr);
			f3 e{0, 0, 0};
			if (sf.emissive) e = shade_emission(sc, sf, s, best, bounce, mis);
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
			if (!shade_continue<GGX>(sf, &s, acc, seed, bounce)) { counters[3]++; break; }
		}
	}
	};
	if (flags & B2R_FLAG_GGX) trace_all(std::true_type{}); else trace_all(std::false_type{});
	return 0;
}

// flatten_bvh tap: out may be null to size
int hc_flatten(const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* prims, uint32_t n_prims, void* out, uint32_t* n_wide, uint32_t* max_stack, const float* box6) {
	const OriginBox ob = origin_box_of(prims, n_prims, box6, nullptr, 0);
	WideBvh w; flatten_bvh(nodes, n_nodes, prims, n_prims, w, &ob);
	*n_wide = static_cast<uint32_t>(w.nodes.size()); *max_stack = w.max_stack;
	if (out) std::memcpy(out, w.nodes.data(), w.nodes.size() * sizeof(WideNode));
	return 0;
}

// refit tap (b2r_refit_scene's host twin): the traversal tree (reference_tree = 0) or the flattened reference tree of the spheres
// prims_a, then refit_wide() with prims_b (same order). wide_out may be null to size; cost = sum of inner-slot half areas before / after.
// remap (may be null): prims_b is in a new order, remap[index in prims_a] = index in prims_b of the same sphere.
// Optionally traces rays through the refitted tree (closest hit; prim_out = index into prims_b or -1).
// box6 (may be null): the origin box to size the leaves for (both the build and the refit); default: the library's rule over the spheres
// of the final tree plus the origins of `rays`.
int hc_refit(const b2r_sphere* prims_a, const b2r_bvh_node* nodes_a, uint32_t n_nodes, const b2r_sphere* prims_b, const uint32_t* remap, uint32_t n, void* wide_out, uint32_t* n_wide,
             double cost[2], const float* rays, uint32_t n_rays, float* tfar_out, int32_t* prim_out, const float* box6) {
	WideBvh w;
	float ro[6]; if (n_rays) ray_origin_bounds(rays, n_rays, ro);
	const OriginBox ob_a = origin_box_of(prims_a, n, box6, n_rays ? ro : nullptr, n_rays ? 2u : 0u);
	if (n_nodes == 0) { std::vector<b2r_bvh_node> tree; build_traversal_tree(prims_a, n, tree); flatten_bvh(tree.data(), static_cast<uint32_t>(tree.size()), prims_a, n, w, &ob_a); }
	else flatten_bvh(nodes_a, n_nodes, prims_a, n, w, &ob_a);
	*n_wide = static_cast<uint32_t>(w.nodes.size());
	if (!wide_out && !n_rays) return 0;
	cost[0] = w.cost;
	if (prims_b) {  // null: the tree as flatten_bvh left it
		std::vector<float4> packed(n);
		for (uint32_t i = 0; i < n; i++) packed[i] = make_float4(prims_b[i].position[0], prims_b[i].position[1], prims_b[i].position[2], prims_b[i].radius_sq);
		refit_wide(w, packed.data(), remap, origin_box_of(prims_b, n, box6, n_rays ? ro : nullptr, n_rays ? 2u : 0u));
	}
	cost[1] = w.cost;
	if (wide_out) std::memcpy(wide_out, w.nodes.data(), w.nodes.size() * sizeof(WideNode));
	uint32_t cs = 0, cb = 0;
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		traverse_closest<false>(w.nodes.data(), w.tn_bits, Ray{r[0], r[1], r[2], r[3], r[4], r[5]}, tfar_out + i, prim_out + i, &cs, &cb);
	}
	return 0;
}
// build_packed_tree tap: the host twin of the tree b2r_upload_scene builds on the GPU with B2R_FLAG_GPU_TREE. out may be null to size.
int hc_packed_tree(const b2r_sphere* prims, uint32_t n, const float* box6, void* out, uint32_t* n_wide, uint32_t* max_stack) {
	const OriginBox ob = origin_box_of(prims, n, box6, nullptr, 0);
	WideBvh w; build_packed_tree(prims, n, w, &ob);
	*n_wide = static_cast<uint32_t>(w.nodes.size()); *max_stack = w.max_stack;
	if (out) std::memcpy(out, w.nodes.data(), w.nodes.size() * sizeof(WideNode));
	return 0;
}
// build_sweep_tree tap: the host twin of the tree b2r_upload_scene builds on the GPU with B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH. Returns 1 when
// the tree would be too deep (the library then builds the packed tree).
int hc_sweep_tree(const b2r_sphere* prims, uint32_t n, const float* box6, void* out, uint32_t* n_wide, uint32_t* max_stack) {
	const OriginBox ob = origin_box_of(prims, n, box6, nullptr, 0);
	WideBvh w; if (!build_sweep_tree(prims, n, w, &ob)) return 1;
	*n_wide = static_cast<uint32_t>(w.nodes.size()); *max_stack = w.max_stack;
	if (out) std::memcpy(out, w.nodes.data(), w.nodes.size() * sizeof(WideNode));
	return 0;
}
int hc_sweep3_tree(const b2r_sphere* prims, uint32_t n, const float* box6, void* out, uint32_t* n_wide, uint32_t* max_stack) {
	const OriginBox ob = origin_box_of(prims, n, box6, nullptr, 0);
	WideBvh w; if (!build_sweep3_tree(prims, n, w, &ob)) return 1;
	*n_wide = static_cast<uint32_t>(w.nodes.size()); *max_stack = w.max_stack;
	if (out) std::memcpy(out, w.nodes.data(), w.nodes.size() * sizeof(WideNode));
	return 0;
}
// the sort key of build_packed_tree / k_morton_keys (b2r_shade.h: morton_key) for sphere centres inside [lo, hi]
int hc_curve_keys(const b2r_sphere* prims, uint32_t n, const float lo[3], const float hi[3], uint32_t* keys_out) {
	std::vector<uint32_t> keys; morton_keys(prims, n, lo, hi, keys);
	std::memcpy(keys_out, keys.data(), n * sizeof(uint32_t));
	return 0;
}
// validate_reference_bvh tap (what b2r_upload_scene checks before it flattens a caller's node array)
int hc_validate(const b2r_bvh_node* nodes, uint32_t n_nodes, uint32_t n_prims) { return validate_reference_bvh(nodes, n_nodes, n_prims) ? 1 : 0; }
// match_prims_to_geometry tap: geom_of_prim[n]; returns 1 when prims is a permutation of geometry
int hc_match(const b2r_sphere* prims, const b2r_sphere* geometry, uint32_t n, uint32_t* geom_of_prim) {
	std::vector<uint32_t> m; if (!match_prims_to_geometry(prims, geometry, n, m)) return 0;
	std::memcpy(geom_of_prim, m.data(), n * sizeof(uint32_t)); return 1;
}
// brute-force closest hit over spheres in order (ties to the lowest index, BVH.hpp:265) for the same rays
void hc_closest_brute(const b2r_sphere* prims, uint32_t n, const float* rays, uint32_t n_rays, float* tfar_out, int32_t* prim_out) {
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		float best = FLT_MAX; int32_t prim = -1;
		for (uint32_t j = 0; j < n; j++) { float d; if (sphere_hit_closest(prims[j].position[0], prims[j].position[1], prims[j].position[2], prims[j].radius_sq, r[0], r[1], r[2], r[3], r[4], r[5], &d) && d < best) { best = d; prim = static_cast<int32_t>(j); } }
		tfar_out[i] = best; prim_out[i] = prim;
	}
}

// brute-force any hit over spheres in order along [0, tfar) (Traverse_shadow without a tree, BVH.hpp:290-305): occ_out[i] = 0 / 1
void hc_any_brute(const b2r_sphere* prims, uint32_t n, const float* rays, const float* tfar, uint32_t n_rays, uint8_t* occ_out) {
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		bool occ = false;
		for (uint32_t j = 0; j < n && !occ; j++) occ = sphere_hit_any(prims[j].position[0], prims[j].position[1], prims[j].position[2], prims[j].radius_sq, r[0], r[1], r[2], r[3], r[4], r[5], tfar[i]);
		occ_out[i] = occ ? 1 : 0;
	}
}
// the same with the scalar-tail formula of the closest-hit loop (BVH.hpp:270-286), spheres in order: what B2R_FLAG_REFERENCE_EXACT's tail rays get
void hc_closest_brute_scalar(const b2r_sphere* prims, uint32_t n, const float* rays, uint32_t n_rays, float* tfar_out, int32_t* prim_out) {
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		float best = FLT_MAX; int32_t prim = -1;
		for (uint32_t j = 0; j < n; j++) sphere_closest_scalar_update(prims[j].position[0], prims[j].position[1], prims[j].position[2], prims[j].radius_sq, static_cast<int32_t>(j), r[0], r[1], r[2], r[3], r[4], r[5], &best, &prim);
		tfar_out[i] = best; prim_out[i] = prim;
	}
}

// scalar taps of csrc/b2r_math.h for function-level comparison with the oracle
uint32_t hc_hash_2d(uint32_t x, uint32_t y) { return hash_2d(x, y); }
uint32_t hc_hash_u32(uint32_t x) { return hash_u32(x); }
void hc_pcg3(uint32_t state, float out[2], uint32_t* bounded, uint32_t range, uint32_t* state_out) { Pcg r{state}; out[0] = r.next_unit(); out[1] = r.next_unit(); *bounded = r.next_below(range); *state_out = r.state; }
void hc_sincos(float x, float* s, float* c) { sincos_poly(x, s, c); }
float hc_asin(float x) { return asin_poly(x); }
float hc_atan2(float y, float x) { return atan2_poly(y, x); }
void hc_hemisphere(float u0, float u1, float out[3]) { f3 v = cosine_hemisphere(u0, u1); out[0] = v.x; out[1] = v.y; out[2] = v.z; }
void hc_tangent(const float n[3], float out_wxyz[4]) { TangentQuat q = tangent_frame(f3{n[0], n[1], n[2]}); out_wxyz[0] = q.w; out_wxyz[1] = q.x; out_wxyz[2] = q.y; out_wxyz[3] = 0.0f; }
void hc_to_local(const float q[4], const float v[3], float out[3]) { f3 r = frame_to_local(TangentQuat{q[0], q[1], q[2]}, f3{v[0], v[1], v[2]}); out[0] = r.x; out[1] = r.y; out[2] = r.z; }
void hc_to_world(const float q[4], const float v[3], float out[3]) { f3 r = frame_to_world(TangentQuat{q[0], q[1], q[2]}, f3{v[0], v[1], v[2]}); out[0] = r.x; out[1] = r.y; out[2] = r.z; }
void hc_onb(const float n[3], float out[6]) { f3 a, b; branchless_onb(f3{n[0], n[1], n[2]}, &a, &b); out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = b.x; out[4] = b.y; out[5] = b.z; }
void hc_sample_sphere(const float wc[3], float s2, float cd, float r2, float u0, float u1, float out[5]) {
	float d, p; f3 L = sample_sphere_cone(f3{wc[0], wc[1], wc[2]}, s2, cd, r2, u0, u1, &d, &p); out[0] = L.x; out[1] = L.y; out[2] = L.z; out[3] = d; out[4] = p;
}
float hc_sphere_pdf(float r2, float d2) { return sphere_light_pdf(r2, d2); }
float hc_power(float f, float g) { return power_heuristic(f, g); }
float hc_power_over_f(float f, float g) { return power_heuristic_over_f(f, g); }
float hc_median5(const float v[5]) { return median_of_5(v[0], v[1], v[2], v[3], v[4]); }
void hc_tonemap(float rgb[3]) { aces_tonemap(rgb, rgb + 1, rgb + 2); }
float hc_median8(const float v[8]) { return median_of_8(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]); }
// closest / any sphere tests: returns 1 and the distance when the candidate is valid
int hc_sphere_closest(const float s[4], const float ray[6], float* d) { return sphere_hit_closest(s[0], s[1], s[2], s[3], ray[0], ray[1], ray[2], ray[3], ray[4], ray[5], d) ? 1 : 0; }
// closest hit over n spheres {c.xyz, r^2} with the scalar-tail formula (BVH.hpp:270-286), all spheres in order
void hc_closest_scalar(const float* spheres4, uint32_t n, const float ray[6], float* best, int32_t* prim) {
	*best = FLT_MAX; *prim = -1;
	for (uint32_t j = 0; j < n; j++) sphere_closest_scalar_update(spheres4[4 * j], spheres4[4 * j + 1], spheres4[4 * j + 2], spheres4[4 * j + 3], static_cast<int32_t>(j), ray[0], ray[1], ray[2], ray[3], ray[4], ray[5], best, prim);
}
int hc_sphere_any(const float s[4], const float ray[6], float tfar) { return sphere_hit_any(s[0], s[1], s[2], s[3], ray[0], ray[1], ray[2], ray[3], ray[4], ray[5], tfar) ? 1 : 0; }

}  // extern "C"

// ---- deterministic traversal taps: every tree the library can trace, the walks the kernels run, and no environment variables.
// Tree kinds of the taps below (the spheres `prims` are in BVH order, as uploaded):
enum HcTree { HC_REFERENCE = 0,  // the caller's reference topology (nodes) flattened: B2R_FLAG_REFERENCE_TREE
              HC_SAH = 1,        // the traversal SAH tree libb2r builds by default
              HC_PACKED = 2,     // the packed tree (B2R_FLAG_GPU_TREE), host twin
              HC_SWEEP = 3,      // the curve sweep tree (B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH), host twin
              HC_SWEEP3 = 4,     // the three-axis sweep tree (B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH3), host twin
              HC_REFIT = 5 };    // the traversal SAH tree of `prims`, refitted to `moved` (same order): b2r_refit_scene's host twin
// Builds tree `kind` for the spheres the rays are traced against (prims, or moved for HC_REFIT). The origin box: box6 when given, else the
// library's rule over the spheres plus the finite ray origins (what b2r_trace_* grows the box to). Returns 0, 1 when a sweep tree would be
// too deep, or B2R_ERR_ARG / B2R_ERR_BVH.
static int hc_tree(int kind, const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* moved, uint32_t n,
                   const float* box6, const float* rays, uint32_t n_rays, WideBvh& w) {
	float pts[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
	for (uint32_t i = 0; i < n_rays; i++) for (int k = 0; k < 3; k++) { const float v = rays[6 * static_cast<size_t>(i) + k]; if (v == v && fabsf(v) <= FLT_MAX) { pts[k] = fminf(pts[k], v); pts[3 + k] = fmaxf(pts[3 + k], v); } }
	const bool have_pts = pts[0] <= pts[3];
	const b2r_sphere* target = kind == HC_REFIT ? moved : prims;
	if (!target) return B2R_ERR_ARG;
	const OriginBox ob = origin_box_of(target, n, box6, have_pts ? pts : nullptr, have_pts ? 2u : 0u);
	switch (kind) {
	case HC_REFERENCE: if (!nodes) return B2R_ERR_ARG; flatten_bvh(nodes, n_nodes, prims, n, w, &ob); break;
	case HC_SAH: case HC_REFIT: { std::vector<b2r_bvh_node> t; build_traversal_tree(prims, n, t); flatten_bvh(t.data(), static_cast<uint32_t>(t.size()), prims, n, w, &ob); break; }
	case HC_PACKED: build_packed_tree(prims, n, w, &ob); break;
	case HC_SWEEP: if (!build_sweep_tree(prims, n, w, &ob)) return 1; break;
	case HC_SWEEP3: if (!build_sweep3_tree(prims, n, w, &ob)) return 1; break;
	default: return B2R_ERR_ARG;
	}
	if (kind == HC_REFIT) {
		std::vector<float4> packed(n);
		for (uint32_t i = 0; i < n; i++) packed[i] = make_float4(moved[i].position[0], moved[i].position[1], moved[i].position[2], moved[i].radius_sq);
		refit_wide(w, packed.data(), nullptr, ob);
	}
	if (w.max_stack + 3u > static_cast<uint32_t>(kTraversalStack)) return B2R_ERR_BVH;
	return 0;
}
extern "C" {

// closest hit through traverse_closest (tail = 1: TravClosestT with the scalar-tail sphere formula, B2R_FLAG_REFERENCE_EXACT's tail rays).
// Compare with hc_closest_brute / hc_closest_brute_scalar over the same spheres (moved for HC_REFIT).
int hc_trace_closest(int kind, const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* moved, uint32_t n, const float* box6,
                     const float* rays, uint32_t n_rays, int tail, float* tfar_out, int32_t* prim_out) {
	WideBvh w; const int rc = hc_tree(kind, prims, nodes, n_nodes, moved, n, box6, rays, n_rays, w); if (rc) return rc;
	uint32_t cs = 0, cb = 0;
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravClosest t; t.begin(Ray{r[0], r[1], r[2], r[3], r[4], r[5]}, tail != 0);
		while (t.step<false>(w.nodes.data(), w.tn_bits, &cs, &cb)) {}
		tfar_out[i] = t.best; prim_out[i] = t.prim;
	}
	return 0;
}
// any hit along [0, tfar) through traverse_any. origin_prim null: every walk starts at the root; else walk i starts, as k_intersect_shadow's
// does, at the node holding sphere origin_prim[i]'s leaf slot and climbs. Compare with hc_any_brute.
int hc_trace_any(int kind, const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* moved, uint32_t n, const float* box6,
                 const float* rays, const float* tfar, const int32_t* origin_prim, uint32_t n_rays, uint8_t* occ_out) {
	WideBvh w; const int rc = hc_tree(kind, prims, nodes, n_nodes, moved, n, box6, rays, n_rays, w); if (rc) return rc;
	std::vector<uint32_t> parent, leaf_node; hc_link_tables(w, n, parent, leaf_node);
	uint32_t cs = 0, cb = 0;
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		if (origin_prim && (origin_prim[i] < 0 || static_cast<uint32_t>(origin_prim[i]) >= n)) return B2R_ERR_ARG;
		const uint32_t start = origin_prim ? leaf_node[origin_prim[i]] : 0u;
		occ_out[i] = traverse_any<false>(w.nodes.data(), Ray{r[0], r[1], r[2], r[3], r[4], r[5]}, tfar[i], &cs, &cb, parent.data(), start) ? 1 : 0;
	}
	return 0;
}
// the slot boxes of tree `kind` as {lo.xyz, hi.xyz, link} per non-empty slot (7 floats, link as int bits); out may be null to count
int hc_tree_boxes(int kind, const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* moved, uint32_t n, const float* box6,
                  const float* rays, uint32_t n_rays, float* out, uint32_t* n_out) {
	WideBvh w; const int rc = hc_tree(kind, prims, nodes, n_nodes, moved, n, box6, rays, n_rays, w); if (rc) return rc;
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	uint32_t m = 0;
	for (size_t nd = 0; nd < w.nodes.size(); nd++) for (int k = 0; k < 4; k++) {
		const float4 a = wide[nd * 8 + 2 * k], b = wide[nd * 8 + 2 * k + 1];
		if (as_int(b.z) == kEmptyLink) continue;
		if (out) { float* o = out + 7 * static_cast<size_t>(m); o[0] = a.x - b.x; o[1] = a.y - b.y; o[2] = a.z - b.w; o[3] = a.x + b.x; o[4] = a.y + b.y; o[5] = a.z + b.w; o[6] = b.z; }
		m++;
	}
	*n_out = m;
	return 0;
}

}  // extern "C"

// per-ray traversal statistics (steps = wide nodes visited, box and sphere tests) for caller rays: tuning aid
extern "C" int hc_trace_stats(const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* prims, uint32_t n_prims, const float* rays, uint32_t n,
                              uint32_t* steps, uint32_t* boxes, uint32_t* spheres, int32_t* prim_out) {
	WideBvh w;
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	if (n_nodes == 0xffffffffu) build_packed_tree(prims, n_prims, w, &ob);   // the packed tree the GPU builds by itself
	else if (n_nodes == 0xfffffffdu) { if (!build_sweep3_tree(prims, n_prims, w, &ob)) return 1; }  // the three-axis sweep tree
	else if (n_nodes == 0xfffffffeu) { if (!build_sweep_tree(prims, n_prims, w, &ob)) return 1; }  // the sweep tree the GPU builds by itself
	else if (n_nodes == 0) { std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn); flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob); }
	else flatten_bvh(nodes, n_nodes, prims, n_prims, w, &ob);
	for (uint32_t i = 0; i < n; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravClosest t; t.begin(Ray{r[0], r[1], r[2], r[3], r[4], r[5]});
		uint32_t cs = 0, cb = 0, st = 0;
		do { st++; } while (t.step<true>(w.nodes.data(), w.tn_bits, &cs, &cb));
		steps[i] = st; boxes[i] = cb; spheres[i] = cs; prim_out[i] = t.prim;
	}
	return 0;
}

// histogram of visited wide-node indices below `top` (BFS order: the first nodes are the top of the tree): tuning aid
extern "C" int hc_trace_top_share(const b2r_sphere* prims, uint32_t n_prims, const float* rays, uint32_t n, uint32_t top, uint64_t* visits_top, uint64_t* visits_all) {
	std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn);
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	WideBvh w; flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob);
	uint64_t a = 0, b = 0;
	for (uint32_t i = 0; i < n; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravClosest t; t.begin(Ray{r[0], r[1], r[2], r[3], r[4], r[5]});
		uint32_t cs = 0, cb = 0; bool more = true;
		while (more) { b++; if (t.node < top) a++; more = t.step<false>(w.nodes.data(), w.tn_bits, &cs, &cb); }
	}
	*visits_top = a; *visits_all = b;
	return 0;
}

// packet traversal statistics (tuning aid): `n` rays in packets of 32 consecutive rays walk the traversal tree TOGETHER — a node is visited
// when any ray of the packet passes its box within its own best distance; children nearest-first by the packet's minimum entry distance.
// Returns the node visits per packet and checks every ray's closest hit against its own single-ray walk (returns the number of mismatches).
extern "C" int hc_packet_stats(const b2r_sphere* prims, uint32_t n_prims, const float* rays, uint32_t n, uint32_t* visits_per_packet, uint32_t* sphere_tests_per_packet) {
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn);
	WideBvh w; flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob);
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	int bad = 0;
	for (uint32_t p0 = 0; p0 < n; p0 += 32) {
		const uint32_t m = std::min(32u, n - p0);
		TravClosest t[32]; float best[32]; int32_t prim[32];
		for (uint32_t i = 0; i < m; i++) { const float* r = rays + 6 * static_cast<size_t>(p0 + i); t[i].begin(Ray{r[0], r[1], r[2], r[3], r[4], r[5]}); best[i] = FLT_MAX; prim[i] = -1; }
		struct E { uint32_t node; float tn; }; std::vector<E> stack; stack.push_back({0u, 0.0f});
		uint32_t visits = 0, stests = 0;
		while (!stack.empty()) {
			const E e = stack.back(); stack.pop_back();
			float wmax = 0.0f; for (uint32_t i = 0; i < m; i++) wmax = std::max(wmax, best[i]);
			if (e.tn > wmax) continue;
			visits++;
			const float4* nd = wide + static_cast<size_t>(e.node) * 8;
			E kids[4]; int nk = 0;
			for (int k = 0; k < 4; k++) {
				const float4 a = nd[2 * k], b = nd[2 * k + 1]; const int32_t l = as_int(b.z);
				if (l == kEmptyLink) continue;
				float tmin = FLT_MAX; bool any = false;
				for (uint32_t i = 0; i < m; i++) {
					float tnr; bool h; slab(a, b, t[i].ix, t[i].iy, t[i].iz, t[i].nx, t[i].ny, t[i].nz, t[i].ax, t[i].ay, t[i].az, best[i], &tnr, &h);
					if (!h) continue;
					any = true; tmin = std::min(tmin, tnr);
					if (l < 0) { float d; stests++; if (sphere_hit_closest(a.x, a.y, a.z, a.w, t[i].ox, t[i].oy, t[i].oz, t[i].dx, t[i].dy, t[i].dz, &d) && (d < best[i] || (d == best[i] && ~l < prim[i]))) { best[i] = d; prim[i] = ~l; } }
				}
				if (any && l >= 0) kids[nk++] = {static_cast<uint32_t>(l), tmin};
			}
			std::sort(kids, kids + nk, [](const E& x, const E& y) { return x.tn > y.tn; });  // farthest first onto the stack
			for (int k = 0; k < nk; k++) stack.push_back(kids[k]);
		}
		visits_per_packet[p0 / 32] = visits; sphere_tests_per_packet[p0 / 32] = stests;
		for (uint32_t i = 0; i < m; i++) { uint32_t cs = 0, cb = 0; float b1; int32_t p1; const float* r = rays + 6 * static_cast<size_t>(p0 + i);
			traverse_closest<false>(w.nodes.data(), w.tn_bits, Ray{r[0], r[1], r[2], r[3], r[4], r[5]}, &b1, &p1, &cs, &cb); if (p1 != prim[i] || bits(b1) != bits(best[i])) bad++; }
	}
	return bad;
}

// any-hit traversal statistics (tuning aid): node visits per shadow ray with the kernels' order (first hit slot first) and with the nearest
// hit child first; occluded_out from the kernels' order; returns the number of rays on which the two policies disagree (must be 0)
extern "C" int hc_anyhit_stats(const b2r_sphere* prims, uint32_t n_prims, const float* rays, const float* tfar, uint32_t n, uint32_t* steps_slot_order, uint32_t* steps_nearest, uint8_t* occluded_out) {
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn);
	WideBvh w; flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob);
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	int bad = 0;
	for (uint32_t i = 0; i < n; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravBase t; t.arm(Ray{r[0], r[1], r[2], r[3], r[4], r[5]});
		bool occ[2] = {false, false}; uint32_t st[2] = {0, 0};
		for (int policy = 0; policy < 2; policy++) {
			const int mode = policy == 0 ? 0 : (std::getenv("HC_ANYHIT_MODE") ? std::atoi(std::getenv("HC_ANYHIT_MODE")) : 1);
			std::vector<uint32_t> stack; uint32_t node = 0; bool have = true;
			while (have && !occ[policy]) {
				st[policy]++;
				const float4* nd = wide + static_cast<size_t>(node) * 8;
				uint32_t hit[4]; float htn[4]; int nh = 0;
				for (int k = 0; k < 4 && !occ[policy]; k++) {
					const float4 a = nd[2 * k], b = nd[2 * k + 1]; const int32_t l = as_int(b.z);
					float tnr; bool h; slab(a, b, t.ix, t.iy, t.iz, t.nx, t.ny, t.nz, t.ax, t.ay, t.az, tfar[i], &tnr, &h);
					if (!h) continue;
					if (l < 0) { if (sphere_hit_any(a.x, a.y, a.z, a.w, t.ox, t.oy, t.oz, t.dx, t.dy, t.dz, tfar[i])) occ[policy] = true; }
					else { hit[nh] = static_cast<uint32_t>(l); htn[nh] = tnr; nh++; }
				}
				if (occ[policy]) break;
				if (mode == 1 && nh > 1) { int m = 0; for (int k = 1; k < nh; k++) if (htn[k] < htn[m]) m = k; std::swap(hit[0], hit[m]); std::swap(htn[0], htn[m]); }
				if (mode == 2 && nh > 1) { for (int a2 = 0; a2 < nh; a2++) for (int b2 = a2 + 1; b2 < nh; b2++) if (htn[b2] < htn[a2]) { std::swap(hit[a2], hit[b2]); std::swap(htn[a2], htn[b2]); } }
				for (int k = nh - 1; k >= 1; k--) stack.push_back(hit[k]);
				if (nh) node = hit[0]; else if (!stack.empty()) { node = stack.back(); stack.pop_back(); } else have = false;
			}
		}
		if (occ[0] != occ[1]) bad++;
		steps_slot_order[i] = st[0]; steps_nearest[i] = st[1]; occluded_out[i] = occ[0] ? 1 : 0;
	}
	return bad;
}

// any-hit traversal started BELOW the root (tuning aid): a shadow ray leaves a point on sphere `origin_prim`, and in a dense scene its
// occluder is usually a neighbour, so the walk starts at the ancestor `height` levels above the node that holds the origin sphere's leaf
// slot and only falls back to the root (skipping the subtree already searched) when that subtree holds no occluder. The result is the same
// order-independent boolean. steps_root = visits of the walk from the root (nearest hit child first), steps_local = visits of the two-phase walk.
extern "C" int hc_anyhit_local_stats(const b2r_sphere* prims, uint32_t n_prims, const float* rays, const float* tfar, const int32_t* origin_prim, uint32_t n, uint32_t height,
                                     uint32_t* steps_root, uint32_t* steps_local, uint8_t* found_local) {
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn);
	WideBvh w; flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob);
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	std::vector<uint32_t> parent, leaf_node; hc_link_tables(w, n_prims, parent, leaf_node);
	int bad = 0;
	for (uint32_t i = 0; i < n; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravBase t; t.arm(Ray{r[0], r[1], r[2], r[3], r[4], r[5]});
		uint32_t start = leaf_node[origin_prim[i]]; for (uint32_t h = 0; h < height; h++) start = parent[start];
		auto walk = [&](uint32_t from, uint32_t skip, uint32_t* steps) {
			std::vector<uint32_t> stack; uint32_t node = from; bool have = true, occ = false;
			while (have && !occ) {
				(*steps)++;
				const float4* nd = wide + static_cast<size_t>(node) * 8;
				uint32_t hit[4]; float htn[4]; int nh = 0;
				for (int k = 0; k < 4 && !occ; k++) {
					const float4 a = nd[2 * k], b = nd[2 * k + 1]; const int32_t l = as_int(b.z);
					float tnr; bool h; slab(a, b, t.ix, t.iy, t.iz, t.nx, t.ny, t.nz, t.ax, t.ay, t.az, tfar[i], &tnr, &h);
					if (!h) continue;
					if (l < 0) { if (sphere_hit_any(a.x, a.y, a.z, a.w, t.ox, t.oy, t.oz, t.dx, t.dy, t.dz, tfar[i])) occ = true; }
					else if (static_cast<uint32_t>(l) != skip) { hit[nh] = static_cast<uint32_t>(l); htn[nh] = tnr; nh++; }
				}
				if (occ) break;
				if (nh > 1) { int m = 0; for (int k = 1; k < nh; k++) if (htn[k] < htn[m]) m = k; std::swap(hit[0], hit[m]); std::swap(htn[0], htn[m]); }
				for (int k = nh - 1; k >= 1; k--) stack.push_back(hit[k]);
				if (nh) node = hit[0]; else if (!stack.empty()) { node = stack.back(); stack.pop_back(); } else have = false;
			}
			return occ;
		};
		uint32_t sr = 0, sl = 0;
		const bool occ_root = walk(0u, 0xffffffffu, &sr);
		bool occ_local = walk(start, 0xffffffffu, &sl);
		found_local[i] = occ_local ? 1 : 0;
		if (std::getenv("HC_CLIMB")) {  // instead of restarting at the root: climb one level at a time, searching the siblings not yet searched
			uint32_t cur = start;
			while (!occ_local && cur != 0u) { const uint32_t up = parent[cur]; occ_local = walk(up, cur, &sl); cur = up; }
		} else
		if (!occ_local && start != 0u) occ_local = walk(0u, start, &sl);
		if (occ_root != occ_local) bad++;
		steps_root[i] = sr; steps_local[i] = sl;
	}
	return bad;
}

// closest-hit walk started at the node that holds the origin sphere and climbing to the root (tuning aid), against the walk from the root:
// node visits, pushes and pops (culled ones included) per ray. out[6 * i + {0,1,2}] = root walk, {3,4,5} = climbing walk. Returns mismatches.
extern "C" int hc_closest_climb_stats(const b2r_sphere* prims, uint32_t n_prims, const float* rays, const int32_t* origin_prim, uint32_t n, uint32_t* out) {
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn);
	WideBvh w; flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob);
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	std::vector<uint32_t> parent, leaf_node; hc_link_tables(w, n_prims, parent, leaf_node);
	int bad = 0;
	for (uint32_t i = 0; i < n; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravBase t; t.arm(Ray{r[0], r[1], r[2], r[3], r[4], r[5]});
		float bestm[2]; int32_t primm[2];
		for (int mode = 0; mode < 2; mode++) {
			struct E { uint32_t node; float tn; }; std::vector<E> stack; float best = FLT_MAX; int32_t prim = -1; uint32_t st = 0, pushes = 0, pops = 0; bool have = true;
			uint32_t root = mode == 0 ? 0u : leaf_node[origin_prim[i]], skip = 0xffffffffu, node = root;
			while (have) {
				st++;
				const float4* nd = wide + static_cast<size_t>(node) * 8;
				E kids[4]; int nk = 0;
				for (int k = 0; k < 4; k++) {
					const float4 a = nd[2 * k], b = nd[2 * k + 1]; const int32_t l = as_int(b.z);
					float tnr; bool h; slab(a, b, t.ix, t.iy, t.iz, t.nx, t.ny, t.nz, t.ax, t.ay, t.az, best, &tnr, &h);
					if (!h) continue;
					if (l < 0) { float d; if (sphere_hit_closest(a.x, a.y, a.z, a.w, t.ox, t.oy, t.oz, t.dx, t.dy, t.dz, &d) && (d < best || (d == best && ~l < prim))) { best = d; prim = ~l; } }
					else if (static_cast<uint32_t>(l) != skip) kids[nk++] = {static_cast<uint32_t>(l), tnr};
				}
				std::stable_sort(kids, kids + nk, [](const E& x, const E& y) { return x.tn < y.tn; });
				for (int k = nk - 1; k >= 1; k--) if (kids[k].tn <= best) { stack.push_back(kids[k]); pushes++; }
				have = false;
				if (nk && kids[0].tn <= best) { node = kids[0].node; have = true; }
				else while (!stack.empty()) { const E e = stack.back(); stack.pop_back(); pops++; if (e.tn <= best) { node = e.node; have = true; break; } }
				if (!have && root != 0u) { skip = root; root = parent[root]; node = root; have = true; }
			}
			bestm[mode] = best; primm[mode] = prim; out[6 * static_cast<size_t>(i) + 3 * mode] = st; out[6 * static_cast<size_t>(i) + 3 * mode + 1] = pushes; out[6 * static_cast<size_t>(i) + 3 * mode + 2] = pops;
		}
		if (primm[0] != primm[1] || bits(bestm[0]) != bits(bestm[1])) bad++;
	}
	return bad;
}

// closest-hit traversal statistics for push-order policies (tuning aid): mode 0 = the kernels' order (all hit children sorted by entry
// distance), 1 = nearest child next, the others pushed in slot order, 2 = nearest next, the others pushed farthest-slot-first by a single
// compare of the two remaining... Returns mismatching rays against mode 0 (must be 0); steps_out[mode][ray].
extern "C" int hc_closest_order_stats(const b2r_sphere* prims, uint32_t n_prims, const float* rays, uint32_t n, uint32_t* steps0, uint32_t* steps1) {
	float ro[6]; ray_origin_bounds(rays, n, ro);
	const OriginBox ob = origin_box_of(prims, n_prims, nullptr, ro, 2);
	std::vector<b2r_bvh_node> tn; build_traversal_tree(prims, n_prims, tn);
	WideBvh w; flatten_bvh(tn.data(), static_cast<uint32_t>(tn.size()), prims, n_prims, w, &ob);
	const float4* wide = reinterpret_cast<const float4*>(w.nodes.data());
	int bad = 0;
	for (uint32_t i = 0; i < n; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		TravBase t; t.arm(Ray{r[0], r[1], r[2], r[3], r[4], r[5]});
		float bestm[2]; int32_t primm[2];
		for (int mode = 0; mode < 2; mode++) {
			struct E { uint32_t node; float tn; }; std::vector<E> stack; float best = FLT_MAX; int32_t prim = -1; uint32_t node = 0, st = 0; bool have = true;
			while (have) {
				st++;
				const float4* nd = wide + static_cast<size_t>(node) * 8;
				E kids[4]; int nk = 0;
				for (int k = 0; k < 4; k++) {
					const float4 a = nd[2 * k], b = nd[2 * k + 1]; const int32_t l = as_int(b.z);
					float tnr; bool h; slab(a, b, t.ix, t.iy, t.iz, t.nx, t.ny, t.nz, t.ax, t.ay, t.az, best, &tnr, &h);
					if (!h) continue;
					if (l < 0) { float d; if (sphere_hit_closest(a.x, a.y, a.z, a.w, t.ox, t.oy, t.oz, t.dx, t.dy, t.dz, &d) && (d < best || (d == best && ~l < prim))) { best = d; prim = ~l; } }
					else kids[nk++] = {static_cast<uint32_t>(l), tnr};
				}
				if (mode == 0) std::stable_sort(kids, kids + nk, [](const E& x, const E& y) { return x.tn < y.tn; });
				else if (nk > 1) { int m = 0; for (int k = 1; k < nk; k++) if (kids[k].tn < kids[m].tn) m = k; std::swap(kids[0], kids[m]); }
				for (int k = nk - 1; k >= 1; k--) if (kids[k].tn <= best) stack.push_back(kids[k]);
				have = false;
				if (nk && kids[0].tn <= best) { node = kids[0].node; have = true; }
				else while (!stack.empty()) { const E e = stack.back(); stack.pop_back(); if (e.tn <= best) { node = e.node; have = true; break; } }
			}
			bestm[mode] = best; primm[mode] = prim; (mode == 0 ? steps0 : steps1)[i] = st;
		}
		if (primm[0] != primm[1] || bits(bestm[0]) != bits(bestm[1])) bad++;
	}
	return bad;
}
