// ltree_oracle.cpp — TEST HARNESS (compiled by tests/test_light_tree.py, never part of libb2r.so).
//
// The CPU oracle with B2R_FLAG_LIGHT_TREE restated from this repo's definition (DESIGN.md §2; the reference picks its lights uniformly, so no
// reference result exists). The sky restatement (tests/skycheck/sky_oracle.cpp, unchanged) is included, and with it the dielectric and lens
// restatements and the oracle itself, so lens, glass, GGX and the sky combine. The per-tile stream loop is restated once more as
// accumulate_tile_ltree: the sky loop line for line plus the ORC_LIGHT_TREE branches (the light picked by descending the tree with the pick's
// draw, its BVH-order sphere in the self test, the tree pdf in both MIS weights, the sampled direction's local-cosine pdf). Without
// ORC_LIGHT_TREE it is the sky loop (test_light_tree.py checks that bit for bit). The tree's nodes are an input (lt_set_tree: the tests pass
// the host builder's, whose own properties are checked separately); the descent, the pdf, the root-to-leaf paths and the light <-> sphere
// map are worked out here again.
#include "../skycheck/sky_oracle.cpp"

namespace {
constexpr uint32_t ORC_LIGHT_TREE = 64u;

struct LTree {
	std::vector<float> nodes;                 // [n][8] {c.xyz, R^2, E, link bits, 0, 0}
	std::vector<std::vector<uint8_t>> path;   // per light: the branches from the root (0 left, 1 right)
	std::vector<int32_t> bvh_sphere;          // per light: the lowest BVH-order sphere equal to it (position, radius^2, material), -1: none
	std::vector<int32_t> light_of;            // per BVH-order sphere: the light it is, -1: none
};
std::map<const Ctx*, LTree> g_tree;

int32_t node_link(const LTree& t, uint32_t n) { int32_t v; std::memcpy(&v, &t.nodes[8 * n + 5], 4); return v; }
// E / max(|P - c|^2, R^2)
float importance(const LTree& t, uint32_t n, V3 P) {
	const float* a = &t.nodes[8 * n];
	const float dx = P.x - a[0], dy = P.y - a[1], dz = P.z - a[2];
	return a[4] / smax((dx * dx + dy * dy) + dz * dz, a[3]);
}
// probability of the left child (nodes link, link + 1): I_l / (I_l + I_r), 1/2 when the sum is 0 or not finite
float left_prob(const LTree& t, uint32_t link, V3 P) {
	const float a = importance(t, link, P), b = importance(t, link + 1u, P), s = a + b;
	return (s > 0.0f && std::isfinite(s)) ? a / s : 0.5f;
}
int32_t tree_pick(const LTree& t, V3 P, float u, float* pdf) {
	uint32_t n = 0; float p = 1.0f;
	while (node_link(t, n) >= 0) {
		const uint32_t link = static_cast<uint32_t>(node_link(t, n));
		const float pl = left_prob(t, link, P), pr = 1.0f - pl;
		if (pr == 0.0f || (pl > 0.0f && u < pl)) { p = p * pl; u = u / pl; n = link; }  // a branch of probability 0 is never taken
		else { p = p * pr; u = (u - pl) / pr; n = link + 1u; }
		if (u >= 1.0f) u = 0x1.fffffep-1f;
	}
	*pdf = p;
	return ~node_link(t, n);
}
float tree_pdf(const LTree& t, V3 P, int32_t light) {
	uint32_t n = 0; float p = 1.0f;
	for (uint8_t right : t.path[light]) {
		const uint32_t link = static_cast<uint32_t>(node_link(t, n));
		const float pl = left_prob(t, link, P), pr = 1.0f - pl;
		p = p * (right ? pr : pl); n = link + right;
	}
	return p;
}

void accumulate_tile_ltree(Ctx& c, uint32_t LaunchIndex, TileScratch& S, DielScratch& Dl, const SkyTab* sky, const LTree* tree) {
	const uint32_t accumulations = c.accumulations;
	const uint32_t light_count = static_cast<uint32_t>(c.lights.size());
	const bool has_ambient = smax(c.ambient[0], smax(c.ambient[1], c.ambient[2])) > 0.0f;
	// ORC_SKY_LIGHT: p_sky = 1 without sphere lights, 1/2 with them, 0 without a sampled sky (no tables); the spheres' selection pdf (1 - p_sky) / n
	const bool sky_on = (c.flags & ORC_SKY_LIGHT) != 0 && has_ambient && sky != nullptr;
	const float p_sky = !sky_on ? 0.0f : light_count == 0 ? 1.0f : 0.5f;
	const float light_selection_pdf = (c.flags & ORC_SKY_LIGHT) ? (light_count ? (1.0f - p_sky) / static_cast<float>(light_count) : 0.0f) : 1.0f / static_cast<float>(c.lights.size());
	const uint32_t bucket_index = accumulations % c.K;
	const bool mis = !(c.flags & ORC_NO_MIS);
	const bool ggx = (c.flags & ORC_GGX) != 0;
	const bool diel_on = (c.flags & ORC_DIELECTRIC) != 0;
	const bool tree_on = (c.flags & ORC_LIGHT_TREE) != 0 && tree != nullptr;  // ORC_LIGHT_TREE: a sphere light's selection pdf is (1 - p_sky) * tree_pdf
	float* out_r = c.accumulator.data() + (static_cast<size_t>(LaunchIndex) * c.K + bucket_index) * 3 * kTileSize;
	float* out_g = out_r + kTileSize; float* out_b = out_g + kTileSize;
	const int32_t tile_x = kTileRoot * static_cast<int32_t>(LaunchIndex % c.h_tiles);
	const int32_t tile_y = kTileRoot * static_cast<int32_t>(LaunchIndex / c.h_tiles);
	uint64_t n_ext = 0, n_shadow = 0, n_shaded = 0, n_term = 0, n_sphere = 0, n_box = 0, n_dropped = 0;

	Buffer* in = &S.buffers[0]; Buffer* out = &S.buffers[1];
	for (int i = 0; i < kTileSize; i++) {
		in->rr[i] = in->rg[i] = in->rb[i] = 0.0f;
		in->tr[i] = in->tg[i] = in->tb[i] = 1.0f;
		in->pixelID[i] = static_cast<uint32_t>(i);
		S.seed[i] = static_cast<uint32_t>(static_cast<int32_t>((static_cast<size_t>(LaunchIndex) * kTileSize + i) * (c.max_bounces * 2 + 1)));
	}
	for (int ID = 0; ID < kTileSize; ID++) {
		int32_t x = tile_x + ID % kTileRoot, y = tile_y + ID / kTileRoot;
		uint32_t rng_state = hash_2d(accumulations, S.seed[ID]);
		const float camera_samples[2] = {rand_unit_float(&rng_state), rand_unit_float(&rng_state)};
		V3 o, d; generate_ray(c, x, y, camera_samples, &o, &d);  // non-const Ctx: the lens oracle's camera ray
		in->dx[ID] = d.x; in->dy[ID] = d.y; in->dz[ID] = d.z; in->px[ID] = o.x; in->py[ID] = o.y; in->pz[ID] = o.z;
	}
	S.sort_buffer.assign(std::max<size_t>(64, c.material.size() + 2), 0);

	size_t active_rays = kTileSize;
	for (size_t bounce = 0; bounce < c.max_bounces && active_rays > 0; bounce++, std::swap(in, out)) {
		std::memset(S.termination, 0, sizeof S.termination); std::memset(S.has_shadowray, 0, sizeof S.has_shadowray);
		std::memset(S.shadow.occluded, 0, sizeof S.shadow.occluded); std::memset(S.sd.is_emissive, 0, sizeof S.sd.is_emissive);
		std::memset(Dl.is_diel, 0, sizeof Dl.is_diel);
		std::fill(S.sort_buffer.begin(), S.sort_buffer.end(), 0u);
		for (size_t i = 0; i < ((active_rays + 7) / 8) * 8; i++) { S.hit.tfar[i] = FLT_MAX; S.hit.matID[i] = -1; S.hit.primID[i] = -1; }

		n_ext += active_rays;
		traverse(c, *in, S.hit, active_rays, n_sphere, n_box);

		for (size_t ID = 0; ID < active_rays; ID++) {  // closest-hit shader
			const int32_t mat_ID = S.hit.matID[ID];
			if (mat_ID == -1) continue;
			const int32_t prim_ID = S.hit.primID[ID];
			const float depth = S.hit.tfar[ID];
			const V3 D{in->dx[ID], in->dy[ID], in->dz[ID]};
			V3 hit_point{in->px[ID] + D.x * depth, in->py[ID] + D.y * depth, in->pz[ID] + D.z * depth};
			const Sphere& sp = c.bvh.prims[prim_ID];
			V3 N{hit_point.x - sp.px, hit_point.y - sp.py, hit_point.z - sp.pz};
			N = normalize(N);
			const bool leaving = dot(N, D) >= 0.0f;
			if (leaving) N = -N;
			Quat T = tangent_space(N);
			V3 Vlocal = to_local(T, -D);
			S.sd.Px[ID] = hit_point.x + N.x * 1e-4f; S.sd.Py[ID] = hit_point.y + N.y * 1e-4f; S.sd.Pz[ID] = hit_point.z + N.z * 1e-4f;
			S.sd.Vx[ID] = Vlocal.x; S.sd.Vy[ID] = Vlocal.y; S.sd.Vz[ID] = Vlocal.z;
			S.sd.Tx[ID] = T.x; S.sd.Ty[ID] = T.y; S.sd.Tz[ID] = T.z; S.sd.Tw[ID] = T.w;
			const Material& m = c.material[mat_ID];
			if (smax(m.emission[0], smax(m.emission[1], m.emission[2])) > FLT_EPSILON) S.sd.is_emissive[ID] = 1;
			if (!ggx) { S.sd.albedo[ID][0] = m.albedo[0]; S.sd.albedo[ID][1] = m.albedo[1]; S.sd.albedo[ID][2] = m.albedo[2]; }
			else {
				S.sd.albedo[ID][0] = m.F0[0]; S.sd.albedo[ID][1] = m.F0[1]; S.sd.albedo[ID][2] = m.F0[2];
				float alpha = m.roughness; alpha *= alpha;
				S.sd.alpha[ID] = alpha + (1.0f - alpha) * 0.0f;
			}
			if (diel_on && smax(m.transmission[0], smax(m.transmission[1], m.transmission[2])) > 0.0f) {  // ORC_DIELECTRIC
				Dl.is_diel[ID] = 1; Dl.inside[ID] = leaving ? 1 : 0;
				Dl.Qx[ID] = hit_point.x - N.x * 1e-4f; Dl.Qy[ID] = hit_point.y - N.y * 1e-4f; Dl.Qz[ID] = hit_point.z - N.z * 1e-4f;
			}
		}

		size_t miss_count;  // sort_rayID
		{
			uint32_t* sb = S.sort_buffer.data();
			const uint32_t k = static_cast<uint32_t>(c.material.size());
			for (size_t i = 0; i < active_rays; i++) ++sb[1 + S.hit.matID[i]];
			miss_count = sb[0];
			for (uint32_t i = 1; i < k + 1; i++) sb[i] += sb[i - 1];
			for (int32_t i = static_cast<int32_t>(active_rays) - 1; i >= 0; i--) S.RayID[--sb[1 + S.hit.matID[i]]] = static_cast<uint32_t>(i);
		}
		const size_t hit_count = active_rays - miss_count;
		n_shaded += hit_count;

		if (mis && (light_count > 0 || p_sky > 0.0f)) {  // NEE
			size_t shadow_index = 0;
			for (size_t i = 0; i < hit_count; i++) {
				const int32_t ID = static_cast<int32_t>(S.RayID[miss_count + i]);
				if (Dl.is_diel[ID]) continue;  // ORC_DIELECTRIC: a delta BSDF takes no light sample
				uint32_t rng_state = hash_2d(accumulations, S.seed[in->pixelID[ID]] + static_cast<uint32_t>(bounce) * 2);
				const float LightSamples[2] = {rand_unit_float(&rng_state), rand_unit_float(&rng_state)};
				const bool pick_draw = !(c.flags & ORC_SKY_LIGHT) || light_count > 0;
				const float tree_u = (tree_on && pick_draw) ? rand_unit_float(&rng_state) : 0.0f;  // ORC_LIGHT_TREE: the draw rand_bounded_int consumes
				int32_t selected_light = (!tree_on && pick_draw) ? static_cast<int32_t>(rand_bounded_int(&rng_state, light_count)) : 0;
				if (p_sky >= 1.0f || (p_sky > 0.0f && rand_unit_float(&rng_state) < p_sky)) {  // ORC_SKY_LIGHT: a sky sample, four more draws
					const float um = rand_unit_float(&rng_state), uc = rand_unit_float(&rng_state), uy = rand_unit_float(&rng_state), ux = rand_unit_float(&rng_state);
					const uint32_t row = cdf_find(sky->marg.data(), sky->rows, um);
					const uint32_t col = cdf_find(sky->cond.data() + static_cast<size_t>(row) * (sky->cols + 1u), sky->cols, uc);
					const float z0 = border_z(row, sky->rows), z1 = border_z(row + 1u, sky->rows);
					const float dy = z0 + uy * (z1 - z0);
					float sin_phi, cos_phi; fast_sincos(kTwoPi * ((static_cast<float>(col) + ux) / static_cast<float>(sky->cols)) - kPi, &sin_phi, &cos_phi);
					const float rxz = std::sqrt(smax(0.0f, 1.0f - dy * dy));
					const V3 L{rxz * cos_phi, dy, rxz * sin_phi};
					Quat T{S.sd.Tw[ID], S.sd.Tx[ID], S.sd.Ty[ID], S.sd.Tz[ID]};
					V3 Llocal = to_local(T, L);
					if (Llocal.z < 0.0f) continue;
					const int32_t texel = sky_index(c, L.x, L.y, L.z);
					const float* tx = c.hdri.data() + 4 * static_cast<size_t>(texel);
					const float q = p_sky * sky->pdf[texel], drawn = p_sky * sky->pdf[static_cast<size_t>(row) * c.hdri_w + col];
					const float f = kOneOverPi * smax(0.0f, Llocal.z);
					V3 radiance{(tx[0] * c.ambient[0]) * in->tr[ID], (tx[1] * c.ambient[1]) * in->tg[ID], (tx[2] * c.ambient[2]) * in->tb[ID]};
					radiance = radiance * V3{S.sd.albedo[ID][0] * f, S.sd.albedo[ID][1] * f, S.sd.albedo[ID][2] * f};
					radiance = radiance * (mis_weight(q, f) / drawn);
					if (smax(smax(radiance.x, radiance.y), radiance.z) <= 0.0f) continue;
					S.shadow.dx[shadow_index] = L.x; S.shadow.dy[shadow_index] = L.y; S.shadow.dz[shadow_index] = L.z;
					S.shadow.px[shadow_index] = S.sd.Px[ID]; S.shadow.py[shadow_index] = S.sd.Py[ID]; S.shadow.pz[shadow_index] = S.sd.Pz[ID];
					S.shadow.tfar[shadow_index] = FLT_MAX;
					S.shadow.r[shadow_index] = radiance.x; S.shadow.g[shadow_index] = radiance.y; S.shadow.b[shadow_index] = radiance.z;
					S.has_shadowray[ID] = 1;
					++shadow_index;
					continue;
				}
				float tree_sel = 0.0f;
				if (tree_on) { selected_light = tree_pick(*tree, V3{S.sd.Px[ID], S.sd.Py[ID], S.sd.Pz[ID]}, tree_u, &tree_sel); tree_sel = (1.0f - p_sky) * tree_sel; }
				int32_t light_primID = c.lights[selected_light];
				const Sphere& light_prim = c.geometry[light_primID];
				if (tree_on ? tree->bvh_sphere[selected_light] == S.hit.primID[ID] : light_primID == S.hit.primID[ID]) continue;  // ORC_LIGHT_TREE: no Q9
				V3 Wc = V3{light_prim.px, light_prim.py, light_prim.pz} - V3{S.sd.Px[ID], S.sd.Py[ID], S.sd.Pz[ID]};
				float center_dist2 = dot(Wc, Wc);
				if (center_dist2 <= light_prim.radius_sq) continue;
				float center_dist = std::sqrt(center_dist2);
				Wc = Wc * (1.0f / center_dist);
				float sinThetaMax2 = light_prim.radius_sq / center_dist2;
				{
					float NdotW = (2.0f * S.sd.Tw[ID]) * (Wc.z * S.sd.Tw[ID] + Wc.x * S.sd.Ty[ID] - S.sd.Tx[ID] * Wc.y) - Wc.z;
					if (NdotW < 0.0f && sinThetaMax2 < NdotW * NdotW) continue;
				}
				float light_distance, light_pdf;
				V3 L = sample_direction_to_sphere(Wc, sinThetaMax2, center_dist, light_prim.radius_sq, LightSamples[0], LightSamples[1], &light_distance, &light_pdf);
				Quat T{S.sd.Tw[ID], S.sd.Tx[ID], S.sd.Ty[ID], S.sd.Tz[ID]};
				V3 Llocal = to_local(T, L);
				if (Llocal.z < 0.0f) continue;
				const Material& lm = c.material[light_prim.material_ID];
				V3 radiance = V3{lm.emission[0], lm.emission[1], lm.emission[2]} * V3{in->tr[ID], in->tg[ID], in->tb[ID]};
				if (!ggx) {
					float NdotL = smax(0.0f, Llocal.z);
					float f = kOneOverPi * NdotL;
					radiance = radiance * V3{S.sd.albedo[ID][0] * f, S.sd.albedo[ID][1] * f, S.sd.albedo[ID][2] * f};
				} else radiance = radiance * ggx_eval(V3{S.sd.albedo[ID][0], S.sd.albedo[ID][1], S.sd.albedo[ID][2]}, S.sd.alpha[ID], Llocal, V3{S.sd.Vx[ID], S.sd.Vy[ID], S.sd.Vz[ID]});
				light_pdf *= tree_on ? tree_sel : light_selection_pdf;
				float brdf_pdf = ggx ? 0.0f : kOneOverPi * smax(0.0f, Llocal.z);
				radiance = radiance * powerHeuristic_over_f(light_pdf, brdf_pdf);
				if (smax(smax(radiance.x, radiance.y), radiance.z) <= 0.0f) continue;
				S.shadow.dx[shadow_index] = L.x; S.shadow.dy[shadow_index] = L.y; S.shadow.dz[shadow_index] = L.z;
				S.shadow.px[shadow_index] = S.sd.Px[ID]; S.shadow.py[shadow_index] = S.sd.Py[ID]; S.shadow.pz[shadow_index] = S.sd.Pz[ID];
				S.shadow.tfar[shadow_index] = light_distance;
				S.shadow.r[shadow_index] = radiance.x; S.shadow.g[shadow_index] = radiance.y; S.shadow.b[shadow_index] = radiance.z;
				S.has_shadowray[ID] = 1;
				++shadow_index;
			}
			n_shadow += shadow_index;
			traverse_shadow(c, S.shadow, shadow_index, n_sphere, n_box);
			for (size_t i = miss_count, shadow_ID = 0; i < active_rays; i++) {
				const int32_t ID = static_cast<int32_t>(S.RayID[i]);
				if (S.has_shadowray[ID]) {
					if (!S.shadow.occluded[shadow_ID]) { in->rr[ID] += S.shadow.r[shadow_ID]; in->rg[ID] += S.shadow.g[shadow_ID]; in->rb[ID] += S.shadow.b[shadow_ID]; }
					++shadow_ID;
				}
			}
		}
		if (mis && bounce > 0) {  // emissive primitive hit
			for (size_t ID = 0; ID < active_rays; ID++) {
				if (!S.sd.is_emissive[ID]) continue;
				V3 throughput{in->tr[ID], in->tg[ID], in->tb[ID]};
				const Sphere& light_prim = c.bvh.prims[S.hit.primID[ID]];
				const float radius2 = light_prim.radius_sq;
				const float depth = S.hit.tfar[ID];
				const float NdotV = S.sd.Vz[ID];
				float center_dist2 = depth * (depth + NdotV * (2.0f * std::sqrt(radius2))) + radius2;
				// ORC_DIELECTRIC: pdf < 0 marks a path continued from a dielectric (delta) surface: no light sample competed, weight 1
				float sel = light_selection_pdf;
				if (tree_on) {  // ORC_LIGHT_TREE: the hit sphere's tree pdf at the ray's origin; 0 when it is not a light
					const int32_t l = tree->light_of[S.hit.primID[ID]];
					sel = l < 0 ? 0.0f : (1.0f - p_sky) * tree_pdf(*tree, V3{in->px[ID], in->py[ID], in->pz[ID]}, l);
				}
				float weight = (diel_on && in->pdf[ID] < 0.0f) ? 1.0f : powerHeuristic(in->pdf[ID], sel * spherePdf(radius2, center_dist2));
				throughput = throughput * weight;
				const float* em = c.material[S.hit.matID[ID]].emission;
				in->rr[ID] += throughput.x * em[0]; in->rg[ID] += throughput.y * em[1]; in->rb[ID] += throughput.z * em[2];
			}
		} else if (mis) {
			for (size_t ID = 0; ID < active_rays; ID++) {
				if (!S.sd.is_emissive[ID]) continue;
				const float* em = c.material[S.hit.matID[ID]].emission;
				in->rr[ID] += em[0]; in->rg[ID] += em[1]; in->rb[ID] += em[2];
			}
		} else {
			for (size_t ID = 0; ID < active_rays; ID++) {
				if (!S.sd.is_emissive[ID]) continue;
				const float* em = c.material[S.hit.matID[ID]].emission;
				in->rr[ID] += in->tr[ID] * em[0]; in->rg[ID] += in->tg[ID] * em[1]; in->rb[ID] += in->tb[ID] * em[2];
			}
		}
		size_t output_index = 0;  // BRDF sampling
		if (bounce < c.max_bounces - 1) {
			for (size_t i = 0; i < hit_count; i++) {
				const int32_t ID = static_cast<int32_t>(S.RayID[miss_count + i]);
				uint32_t rng_state = hash_2d(accumulations, S.seed[in->pixelID[ID]] + static_cast<uint32_t>(bounce) * 2 + 1);
				const float brdf_samples[2] = {rand_unit_float(&rng_state), rand_unit_float(&rng_state)};
				V3 sdir, estimator, origin{S.sd.Px[ID], S.sd.Py[ID], S.sd.Pz[ID]};
				if (Dl.is_diel[ID]) {  // ORC_DIELECTRIC: the first float picks reflection or refraction, the second is unused
					const Material& m = c.material[S.hit.matID[ID]];
					const float eta = 1.0f + m.IOR_minus_one;
					float F;
					if (diel_scatter(V3{S.sd.Vx[ID], S.sd.Vy[ID], S.sd.Vz[ID]}, Dl.inside[ID] ? eta : 1.0f / eta, brdf_samples[0], &sdir, &F)) estimator = V3{1.0f, 1.0f, 1.0f};
					else { estimator = V3{m.transmission[0], m.transmission[1], m.transmission[2]}; origin = V3{Dl.Qx[ID], Dl.Qy[ID], Dl.Qz[ID]}; }
				}
				else if (!ggx) { sdir = hemisphere(brdf_samples[0], brdf_samples[1]); estimator = V3{S.sd.albedo[ID][0], S.sd.albedo[ID][1], S.sd.albedo[ID][2]}; }
				else ggx_sample(V3{S.sd.albedo[ID][0], S.sd.albedo[ID][1], S.sd.albedo[ID][2]}, S.sd.alpha[ID], V3{S.sd.Vx[ID], S.sd.Vy[ID], S.sd.Vz[ID]}, brdf_samples[0], brdf_samples[1], &sdir, &estimator);
				V3 throughput{in->tr[ID], in->tg[ID], in->tb[ID]};
				throughput = throughput * estimator;
				{  // Russian roulette (Q13): the stream's third float
					float q = 1.0f - smax(throughput.x, smax(throughput.y, throughput.z));
					if (rand_unit_float(&rng_state) < q) { S.termination[ID] = 1; continue; }
					throughput = throughput * (1.0f / smax(FLT_EPSILON, 1.0f - q));
				}
				Quat T{S.sd.Tw[ID], S.sd.Tx[ID], S.sd.Ty[ID], S.sd.Tz[ID]};
				const float local_z = sdir.z;
				sdir = to_world(T, sdir);
				out->px[output_index] = origin.x; out->py[output_index] = origin.y; out->pz[output_index] = origin.z;
				out->dx[output_index] = sdir.x; out->dy[output_index] = sdir.y; out->dz[output_index] = sdir.z;
				out->tr[output_index] = throughput.x; out->tg[output_index] = throughput.y; out->tb[output_index] = throughput.z;
				out->rr[output_index] = in->rr[ID]; out->rg[output_index] = in->rg[ID]; out->rb[output_index] = in->rb[ID];
				out->pixelID[output_index] = in->pixelID[ID];
				// ORC_SKY_LIGHT with the sky sampled: the density the direction was drawn with (local cosine), not Q10's world-space one
				// ORC_LIGHT_TREE with sphere lights: likewise
				out->pdf[output_index] = Dl.is_diel[ID] ? -1.0f : ggx ? 0.0f : kOneOverPi * smax(0.0f, (p_sky > 0.0f || (tree_on && light_count > 0)) ? local_z : sdir.z);
				output_index++;
			}
		} else {
			n_dropped += hit_count;  // Q11
		}
		for (size_t i = 0; i < miss_count; i++) S.termination[S.RayID[i]] = 1;  // miss shader
		if (has_ambient) {
			for (size_t i = 0; i < miss_count; i++) {
				const int32_t ID = static_cast<int32_t>(S.RayID[i]);
				V3 sky_rad = sky_eval(c, in->dx[ID], in->dy[ID], in->dz[ID]);
				if (c.flags & ORC_SKY_LIGHT) {  // per channel (no Q14), weighted against the sky's light samples
					const float w = (bounce == 0 || in->pdf[ID] < 0.0f || p_sky <= 0.0f) ? 1.0f
					              : mis_weight(in->pdf[ID], p_sky * sky->pdf[sky_index(c, in->dx[ID], in->dy[ID], in->dz[ID])]);
					in->rr[ID] += (in->tr[ID] * sky_rad.x) * w; in->rg[ID] += (in->tg[ID] * sky_rad.y) * w; in->rb[ID] += (in->tb[ID] * sky_rad.z) * w;
				} else { in->rr[ID] += in->tr[ID] * sky_rad.x; in->rg[ID] += in->tr[ID] * sky_rad.y; in->rb[ID] += in->tr[ID] * sky_rad.z; }
			}
		}
		for (size_t ID = 0; ID < active_rays; ID++) {  // accumulation
			if (!S.termination[ID]) continue;
			const uint32_t px = in->pixelID[ID];
			out_r[px] += in->rr[ID]; out_g[px] += in->rg[ID]; out_b[px] += in->rb[ID];
			n_term++;
		}
		active_rays = output_index;
	}
	c.counters.extension_rays += n_ext; c.counters.shadow_rays += n_shadow; c.counters.shaded_hits += n_shaded;
	c.counters.terminated += n_term; c.counters.sphere_tests += n_sphere; c.counters.box_tests += n_box; c.counters.dropped += n_dropped;
}
}  // namespace

extern "C" {
// the light tree of context c: nodes[n_nodes][8] as b2r_read_light_tree returns them (null: none). Call after orc_set_scene.
void lt_set_tree(const Ctx* c, const float* nodes, uint32_t n_nodes) {
	if (!nodes) { g_tree.erase(c); return; }
	LTree& t = g_tree[c];
	t.nodes.assign(nodes, nodes + 8 * static_cast<size_t>(n_nodes));
	t.path.assign(c->lights.size(), {});
	std::vector<std::pair<uint32_t, std::vector<uint8_t>>> work{{0u, {}}};
	while (!work.empty()) {
		auto [n, p] = work.back(); work.pop_back();
		const int32_t link = node_link(t, n);
		if (link < 0) { t.path[~link] = p; continue; }
		auto l = p, r = p; l.push_back(0); r.push_back(1);
		work.push_back({static_cast<uint32_t>(link), l}); work.push_back({static_cast<uint32_t>(link) + 1u, r});
	}
	auto same = [](const Sphere& a, const Sphere& b) { return std::memcmp(&a, &b, 20) == 0; };
	t.bvh_sphere.assign(c->lights.size(), -1); t.light_of.assign(c->bvh.prims.size(), -1);
	for (size_t l = 0; l < c->lights.size(); l++)
		for (size_t p = 0; p < c->bvh.prims.size(); p++)
			if (same(c->bvh.prims[p], c->geometry[c->lights[l]])) { t.bvh_sphere[l] = static_cast<int32_t>(p); t.light_of[p] = static_cast<int32_t>(l); break; }
}
// sk_accumulate with the loop above
void lt_accumulate(Ctx* c, uint32_t n_samples, int threads) {
	if (threads < 1) threads = 1;
	const size_t n_tiles = static_cast<size_t>(c->h_tiles) * c->v_tiles;
	auto it = g_sky.find(c); const SkyTab* sky = it == g_sky.end() ? nullptr : &it->second;
	auto jt = g_tree.find(c); const LTree* tree = jt == g_tree.end() ? nullptr : &jt->second;
	for (uint32_t s = 0; s < n_samples; s++) {
		++c->accumulations;
		std::atomic<size_t> next{0};
		auto worker = [&] {
			auto S = std::make_unique<TileScratch>(); auto Dl = std::make_unique<DielScratch>();
			for (size_t i; (i = next.fetch_add(1)) < n_tiles;) accumulate_tile_ltree(*c, static_cast<uint32_t>(i), *S, *Dl, sky, tree);
		};
		std::vector<std::thread> pool;
		for (int t = 1; t < threads; t++) pool.emplace_back(worker);
		worker();
		for (auto& t : pool) t.join();
	}
}
}  // extern "C"
