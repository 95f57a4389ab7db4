// climb_taps.cpp — TEST HARNESS (compiled by tests/test_closest_climb.py with the host check's flags, never part of libb2r.so).
//
// The closest-hit walk k_intersect_closest runs for secondary rays — TravClosestT started at the node that holds the ray's origin sphere and
// climbing through parent[] (csrc/b2r_shade.h) — on the CPU, for the CPU-only test tier. The host check (tests/hostcheck/hostcheck.cpp,
// unchanged) is included whole, so its tree kinds (hc_tree), link tables (hc_link_tables) and brute-force taps are available here too.
#include "../hostcheck/hostcheck.cpp"

extern "C" {

// closest hit of every ray through the kernels' TravClosestT on tree `kind` (as hc_trace_closest; tail = 1: the scalar-tail sphere formula).
// origin_prim null: every walk starts at the root; else walk i starts at the node holding sphere origin_prim[i] (BVH order; -1 = the root),
// as k_intersect_closest's do, and climbs. counts (may be null): [3 * i + {0, 1, 2}] = node visits, sphere tests, box tests of ray i.
int cc_trace_closest(int kind, const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* moved, uint32_t n, const float* box6,
                     const float* rays, uint32_t n_rays, int tail, const int32_t* origin_prim, float* tfar_out, int32_t* prim_out, uint32_t* counts) {
	WideBvh w; const int rc = hc_tree(kind, prims, nodes, n_nodes, moved, n, box6, rays, n_rays, w); if (rc) return rc;
	std::vector<uint32_t> parent, leaf_node; hc_link_tables(w, n, parent, leaf_node);
	for (uint32_t i = 0; i < n_rays; i++) {
		const float* r = rays + 6 * static_cast<size_t>(i);
		if (origin_prim && origin_prim[i] >= static_cast<int32_t>(n)) return B2R_ERR_ARG;
		const uint32_t start = origin_prim && origin_prim[i] >= 0 ? leaf_node[origin_prim[i]] : 0u;
		TravClosest t; t.begin(Ray{r[0], r[1], r[2], r[3], r[4], r[5]}, tail != 0, start, parent.data());
		uint32_t cs = 0, cb = 0, visits = 0;
		do { visits++; } while (t.step<true>(w.nodes.data(), w.tn_bits, &cs, &cb, parent.data()));
		tfar_out[i] = t.best; prim_out[i] = t.prim;
		if (counts) { counts[3 * static_cast<size_t>(i)] = visits; counts[3 * static_cast<size_t>(i) + 1] = cs; counts[3 * static_cast<size_t>(i) + 2] = cb; }
	}
	return 0;
}

}  // extern "C"
