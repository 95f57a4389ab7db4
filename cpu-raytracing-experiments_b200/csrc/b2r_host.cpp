// b2r_host.cpp — host-side scene preparation (no CUDA): the reference's SAH sweep BVH with bit-identical node and
// leaf order (BVH.hpp:90-206), the 4-wide flattening for the GPU, the light list (Scene.hpp:12-16) and the camera
// set-up (Camera.hpp:21-32,47-50). The reference builds its BVH on one host thread; here the same algorithm runs on all host cores with
// the node order of the serial one (every index follows from the subtree sizes), and a second tree is built for traversal.
#include "b2r_host.h"
#include "b2r_shade.h"

#include <algorithm>
#include <array>
#include <atomic>
#include <thread>
#include <cmath>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <string>
#include <numeric>
#include <cstdio>

namespace b2r {
namespace {

struct Box { float lo[3], hi[3]; };

inline Box void_box() {  // Node() default: min = +FLT_MAX, max = -FLT_MAX (BVH.hpp:28-29)
	return Box{{FLT_MAX, FLT_MAX, FLT_MAX}, {-FLT_MAX, -FLT_MAX, -FLT_MAX}};
}
inline void grow(Box& a, const Box& b) {  // Node::operator|= (BVH.hpp:35-39) with glm::min / glm::max
	for (int k = 0; k < 3; k++) { a.lo[k] = sel_min(a.lo[k], b.lo[k]); a.hi[k] = sel_max(a.hi[k], b.hi[k]); }
}
// Node::half_area() (BVH.hpp:58-67). The loop there ends before the x extent is used, so the SAH "area" is just
// extent.y * extent.z (SURVEY Q17). Reproduced because it decides every split.
inline float sah_measure(const Box& b) {
	const float ey = b.hi[1] - b.lo[1], ez = b.hi[2] - b.lo[2];
	return 0.0f + ey * ez;
}
inline int widest_axis(const Box& b) {  // Node::largest_axis (BVH.hpp:48-54)
	const float e[3] = {b.hi[0] - b.lo[0], b.hi[1] - b.lo[1], b.hi[2] - b.lo[2]};
	int best = 0;
	if (e[best] < e[1]) best = 1;
	if (e[best] < e[2]) best = 2;
	return best;
}
inline b2r_bvh_node to_node(const Box& b, uint32_t first, uint32_t count) {
	b2r_bvh_node n;
	for (int k = 0; k < 3; k++) { n.min_bound[k] = b.lo[k]; n.max_bound[k] = b.hi[k]; }
	n.first_id = first; n.prim_count = count;
	return n;
}

}  // namespace

void build_reference_bvh(const b2r_sphere* geometry, uint32_t n, std::vector<b2r_bvh_node>& nodes,
                         std::vector<b2r_sphere>& prims, std::vector<uint32_t>& prim_ids, uint32_t log_cluster_size, float cost_ratio) {
	// SplitHeuristic (BVH.hpp:70-83): prim_count(size) = (size + 2^L - 1) >> L as a float; leaf_cost = half_area * prim_count;
	// non_split_cost = half_area * (prim_count - cost_ratio). The app always passes the defaults (L = 0, ratio 1).
	const auto prim_count = [log_cluster_size](uint32_t size) { return static_cast<float>((static_cast<uint64_t>(size) + (1ull << log_cluster_size) - 1ull) >> log_cluster_size); };
	nodes.clear(); prims.clear(); prim_ids.clear();
	if (n == 0) { nodes.push_back(to_node(void_box(), 0, 0)); return; }
	// per-primitive boxes (Sphere::bounds, Primitives.hpp:13-16) and centroids ((max+min)*0.5, BVH.hpp:55-57)
	std::vector<Box> box(n);
	std::vector<float> centroid[3];
	for (auto& c : centroid) c.resize(n);
	for (uint32_t i = 0; i < n; i++) {
		const float r = sqrtf(geometry[i].radius_sq);
		for (int k = 0; k < 3; k++) {
			box[i].lo[k] = geometry[i].position[k] - r;
			box[i].hi[k] = geometry[i].position[k] + r;
			centroid[k][i] = (box[i].hi[k] + box[i].lo[k]) * 0.5f;
		}
	}
	// three index lists ordered by centroid (BVH.hpp:118-122). The reference's std::ranges::sort leaves tie order
	// implementation-defined (Q19); ties are broken by the lower original index here (== MSVC for n <= 32).
	const unsigned hw = std::thread::hardware_concurrency();
	const unsigned threads = n < 20000u ? 1u : (hw ? (hw > 32u ? 32u : hw) : 1u);
	std::vector<uint32_t> order[3];
	{
		auto sort_axis = [&](int k) {
			order[k].resize(n);
			std::iota(order[k].begin(), order[k].end(), 0u);
			const float* key = centroid[k].data();
			std::stable_sort(order[k].begin(), order[k].end(), [key](uint32_t a, uint32_t b) { return key[a] < key[b]; });
		};
		if (threads > 1) { std::thread t1(sort_axis, 1), t2(sort_axis, 2); sort_axis(0); t1.join(); t2.join(); }
		else for (int k = 0; k < 3; k++) sort_axis(k);
	}

	Box root = void_box();
	for (uint32_t i = 0; i < n; i++) grow(root, box[i]);  // BVH.hpp:125
	// The reference numbers its nodes in the order it creates them: a node's child pair when the node is taken off the work stack,
	// smaller range first (BVH.hpp:190-197). A subtree over c spheres creates exactly 2c-2 nodes, so every pair's index follows from
	// the sizes alone — pair(smaller range) = pair + 2, pair(larger range) = pair + 2 + (2*c_smaller - 2) — and disjoint subtrees can
	// be built by different threads into the pre-sized array with the node order of the serial algorithm, bit for bit.
	nodes.assign(2u * static_cast<size_t>(n) - 1u, to_node(void_box(), 0, 0));
	nodes[0] = to_node(root, 0, 0);

	std::vector<float> suffix_cost[3];     // accum_cost: SAH cost of the right part starting at i (BVH.hpp:154); one array per axis
	for (auto& v : suffix_cost) v.resize(n);
	std::vector<uint8_t> goes_left(n);
	std::vector<uint32_t> scratch(n), scratch2(threads > 1 ? n : 0u);  // windows [begin, end) of a job: disjoint between jobs
	struct Job { uint32_t node, begin, count, pair; };
	auto process = [&](Job first, std::vector<Job>* spill, uint32_t spill_above) {
		std::vector<Job> todo;
		todo.push_back(first);
		while (!todo.empty()) {
			const Job job = todo.back(); todo.pop_back();
			if (job.count <= 1) {  // leaf, always one sphere (BVH.hpp:133-137)
				nodes[job.node].first_id = job.begin; nodes[job.node].prim_count = job.count;
				continue;
			}
			if (spill && job.count <= spill_above && job.node != first.node) { spill->push_back(job); continue; }  // a piece for the thread pool
			const uint32_t begin = job.begin, end = job.begin + job.count;
			const uint32_t pair = job.pair;
			nodes[job.node].first_id = pair;
			Box here; for (int k = 0; k < 3; k++) { here.lo[k] = nodes[job.node].min_bound[k]; here.hi[k] = nodes[job.node].max_bound[k]; }

			// fallback split = median on the widest axis, at the "do not split" cost area*(count-1) (BVH.hpp:144, :80-82)
			uint32_t cut = begin + (job.count + 1) / 2; int cut_axis = widest_axis(here);
			float cut_cost = sah_measure(here) * (prim_count(job.count) - cost_ratio);
			// Per axis: right-to-left sweep (the reference's chunked early exit degenerates into one full sweep, Q18, and its `first_right`
			// guard can never cut the left sweep short), then the left-to-right sweep (BVH.hpp:163-170), which stops once the left cost
			// alone exceeds the bound. The reference runs the axes one after the other against a shrinking bound; the left cost never
			// decreases along a sweep, so nothing behind a stop could have improved the bound, and the result is the first strict minimum
			// in (axis, position) order — which is what merging three independent sweeps against the INITIAL bound gives as well.
			struct AxisCut { float cost; uint32_t cut; bool found; };
			const float bound0 = cut_cost;
			auto sweep = [&](int k) {
				const uint32_t* ids = order[k].data(); float* suffix = suffix_cost[k].data();
				AxisCut best{bound0, 0u, false};
				Box acc = void_box();
				for (uint32_t i = end - 1; i > begin; --i) {
					grow(acc, box[ids[i]]);
					suffix[i] = sah_measure(acc) * prim_count(end - i);
				}
				acc = void_box();
				for (uint32_t i = begin; i + 1 < end; ++i) {
					grow(acc, box[ids[i]]);
					const float left = sah_measure(acc) * prim_count(i + 1 - begin);
					if (left > best.cost) break;
					const float total = left + suffix[i + 1];
					if (total < best.cost) { best.cost = total; best.cut = i + 1; best.found = true; }
				}
				return best;
			};
			AxisCut per_axis[3];
			const bool wide_node = spill != nullptr && job.count >= 65536u;  // only the serial top of the tree fans out per node
			if (wide_node) { std::thread t1([&] { per_axis[1] = sweep(1); }), t2([&] { per_axis[2] = sweep(2); }); per_axis[0] = sweep(0); t1.join(); t2.join(); }
			else for (int k = 0; k < 3; k++) per_axis[k] = sweep(k);
			for (int k = 0; k < 3; k++) if (per_axis[k].found && per_axis[k].cost < cut_cost) { cut = per_axis[k].cut; cut_axis = k; cut_cost = per_axis[k].cost; }
			// keep the other two lists consistent with the chosen cut, preserving their order (BVH.hpp:173-184), and take the child boxes
			// (BVH.hpp:109-113,188: a min / max over the spheres of each side — read here from the list that was cut, whose two sides are
			// already in place; the reference reads list 0, the same two sets). On the serial top of the tree the three passes run side by side.
			Box part[2] = {void_box(), void_box()};
			{
				const uint32_t* ids = order[cut_axis].data();
				for (uint32_t i = begin; i < cut; ++i) goes_left[ids[i]] = 1;
				for (uint32_t i = cut; i < end; ++i) goes_left[ids[i]] = 0;
				auto regroup = [&](int k, uint32_t* spare) {  // spare: a window of (end - begin) entries nobody else uses
					uint32_t* a = order[k].data();
					uint32_t l = begin, r = 0;
					for (uint32_t i = begin; i < end; ++i) { const uint32_t id = a[i]; if (goes_left[id]) a[l++] = id; else spare[r++] = id; }
					std::memcpy(a + l, spare, static_cast<size_t>(r) * sizeof(uint32_t));
				};
				auto child_boxes = [&] {
					for (uint32_t i = begin; i < cut; ++i) grow(part[0], box[ids[i]]);
					for (uint32_t i = cut; i < end; ++i) grow(part[1], box[ids[i]]);
				};
				const int k1 = cut_axis == 0 ? 1 : 0, k2 = cut_axis == 2 ? 1 : 2;
				if (wide_node) { std::thread t1(regroup, k1, scratch.data() + begin), t2(regroup, k2, scratch2.data() + begin); child_boxes(); t1.join(); t2.join(); }
				else { regroup(k1, scratch.data() + begin); regroup(k2, scratch.data() + begin); child_boxes(); }
			}
			const uint32_t first_is_right = sah_measure(part[0]) < sah_measure(part[1]) ? 1u : 0u;
			nodes[pair] = to_node(part[first_is_right], 0, 0);
			nodes[pair + 1u] = to_node(part[1 - first_is_right], 0, 0);
			const uint32_t pb[2] = {begin, cut}, pc[2] = {cut - begin, end - cut};
			const uint32_t bigger = pc[0] < pc[1] ? 1u : 0u;  // index of the larger range
			const uint32_t smaller = 1u - bigger;
			const uint32_t pair_small = pair + 2u, pair_big = pair + 2u + (2u * pc[smaller] - 2u);
			// range r lives in node pair + (r == first_is_right ? 0 : 1)
			todo.push_back({pair + (bigger ^ first_is_right), pb[bigger], pc[bigger], pair_big});
			todo.push_back({pair + (smaller ^ first_is_right), pb[smaller], pc[smaller], pair_small});
		}
	};
	if (threads <= 1) process({0u, 0u, n, 1u}, nullptr, 0u);
	else {
		std::vector<Job> pieces;
		process({0u, 0u, n, 1u}, &pieces, n / (threads * 4u) + 1u);
		std::sort(pieces.begin(), pieces.end(), [](const Job& a, const Job& b) { return a.count > b.count; });
		std::atomic<size_t> next{0};
		auto work = [&] { for (;;) { const size_t k = next.fetch_add(1); if (k >= pieces.size()) break; process(pieces[k], nullptr, 0u); } };
		std::vector<std::thread> pool;
		for (unsigned t = 1; t < threads; t++) pool.emplace_back(work);
		work();
		for (auto& t : pool) t.join();
	}
	prims.resize(n); prim_ids.resize(n);
	for (uint32_t i = 0; i < n; i++) { prim_ids[i] = order[0][i]; prims[i] = geometry[order[0][i]]; }  // BVH.hpp:201-205
}

bool validate_reference_bvh(const b2r_bvh_node* nodes, uint32_t n_nodes, uint32_t n_prims) {
	// What flatten_bvh and the reference's own builder rely on (BVH.hpp:90-206): 2n-1 nodes; an inner node's two children are adjacent
	// and were allocated AFTER it (first_id > own index: no cycles); leaves hold one sphere; every node but the root is some inner
	// node's child exactly once and every sphere sits in exactly one leaf (no shared or orphaned subtrees, no sphere rendered twice).
	if (n_nodes == 0) return false;
	if (n_prims == 0) return n_nodes == 1;
	if (n_nodes != 2 * n_prims - 1) return false;
	std::vector<unsigned char> node_seen(n_nodes, 0), prim_seen(n_prims, 0);
	for (uint32_t i = 0; i < n_nodes; i++) {
		if (nodes[i].prim_count == 0) {
			const uint64_t first = nodes[i].first_id;
			if (first <= i || first + 1 >= n_nodes) return false;
			if (node_seen[first] || node_seen[first + 1]) return false;
			node_seen[first] = node_seen[first + 1] = 1;
		} else {
			if (nodes[i].prim_count != 1 || nodes[i].first_id >= n_prims || prim_seen[nodes[i].first_id]) return false;
			prim_seen[nodes[i].first_id] = 1;
		}
	}
	if (node_seen[0]) return false;
	for (uint32_t i = 1; i < n_nodes; i++) if (!node_seen[i]) return false;
	return true;  // n_prims leaves each with a distinct sphere follows from the counts: (n-1) inner nodes claim 2(n-1) children, the rest are leaves
}

namespace {
inline float surface(const b2r_bvh_node& n) {  // true half surface area: only used to pick which child to open
	const float ex = n.max_bound[0] - n.min_bound[0], ey = n.max_bound[1] - n.min_bound[1], ez = n.max_bound[2] - n.min_bound[2];
	return ex * ey + ey * ez + ez * ex;
}
inline float int_as_float(int32_t v) { float f; std::memcpy(&f, &v, 4); return f; }
}  // namespace

double wide_cost(const WideBvh& t) {
	double sum = 0.0;
	for (const WideNode& w : t.nodes) for (int k = 0; k < 4; k++) {
		int32_t link; std::memcpy(&link, &w.slot[k][6], 4);
		if (link >= 0) { const float4* s = reinterpret_cast<const float4*>(w.slot[k]); sum += static_cast<double>(slot_half_area(s[0], s[1])); }
	}
	return sum;
}

bool match_prims_to_geometry(const b2r_sphere* prims, const b2r_sphere* geometry, uint32_t n, std::vector<uint32_t>& geom_of_prim) {
	// open-addressing table over the 20 bytes that make a sphere (bit patterns, so -0 / NaN need no special case): one slot per DISTINCT
	// sphere, holding the first geometry index with that value; equal spheres hang off it as a list in index order and are handed out
	// first in, first out — linear time however many twins a scene has
	static_assert(offsetof(b2r_sphere, material_ID) == 16, "position, radius_sq, material_ID are the first 20 bytes");
	auto hash = [](const b2r_sphere& s) {
		uint32_t w[5]; std::memcpy(w, &s, 20);
		uint64_t h = 0x9e3779b97f4a7c15ull;
		for (uint32_t v : w) { h ^= v; h *= 0xff51afd7ed558ccdull; h ^= h >> 29; }
		return h;
	};
	uint64_t size = 16; while (size < 2ull * n) size <<= 1;
	const uint64_t mask = size - 1;
	constexpr uint32_t kNone = 0xffffffffu;
	std::vector<uint32_t> table(size, kNone), next_same(n, kNone), last(n), cursor(n);
	for (uint32_t g = 0; g < n; g++) {
		uint64_t at = hash(geometry[g]) & mask;
		for (;; at = (at + 1) & mask) {
			const uint32_t rep = table[at];
			if (rep == kNone) { table[at] = g; last[g] = g; cursor[g] = g; break; }
			if (std::memcmp(&geometry[g], &geometry[rep], 20) == 0) { next_same[last[rep]] = g; last[rep] = g; break; }
		}
	}
	geom_of_prim.assign(n, 0u);
	for (uint32_t i = 0; i < n; i++) {
		uint64_t at = hash(prims[i]) & mask;
		for (;; at = (at + 1) & mask) {
			const uint32_t rep = table[at];
			if (rep == kNone) { geom_of_prim.clear(); return false; }              // a sphere geometry does not have
			if (std::memcmp(&prims[i], &geometry[rep], 20) != 0) continue;
			const uint32_t g = cursor[rep];
			if (g == kNone) { geom_of_prim.clear(); return false; }                // more copies of it than geometry has
			cursor[rep] = next_same[g]; geom_of_prim[i] = g;
			break;
		}
	}
	return true;
}

void sphere_bounds(const b2r_sphere* prims, uint32_t n, float lo[3], float hi[3]) {
	for (int k = 0; k < 3; k++) { lo[k] = FLT_MAX; hi[k] = -FLT_MAX; }
	for (uint32_t i = 0; i < n; i++) {
		const float r = sqrtf(prims[i].radius_sq);
		for (int k = 0; k < 3; k++) { lo[k] = fminf(lo[k], prims[i].position[k] - r); hi[k] = fmaxf(hi[k], prims[i].position[k] + r); }
	}
	if (n == 0) for (int k = 0; k < 3; k++) { lo[k] = 0.0f; hi[k] = 0.0f; }
}
OriginBox origin_box_rule(const float sphere_lo[3], const float sphere_hi[3], const float* extra, uint32_t n_extra) {
	OriginBox ob;
	for (int k = 0; k < 3; k++) {
		float lo = sphere_lo[k], hi = sphere_hi[k];
		for (uint32_t i = 0; i < n_extra; i++) { const float v = extra[3 * static_cast<size_t>(i) + k]; if (v == v) { lo = fminf(lo, v); hi = fmaxf(hi, v); } }
		const float slack = 0.125f * (hi - lo) + 1.0f;
		ob.lo[k] = lo - slack; ob.hi[k] = hi + slack;
	}
	return ob;
}
bool origin_box_holds(const OriginBox& ob, const float* points, uint32_t n_points) {
	for (uint32_t i = 0; i < n_points; i++) for (int k = 0; k < 3; k++) {
		const float v = points[3 * static_cast<size_t>(i) + k];
		if (!(v >= ob.lo[k] && v <= ob.hi[k])) return false;
	}
	return true;
}

void wide_fill_boxes(WideBvh& out, const float4* packed_prims, const OriginBox& ob) {
	float4* wide = reinterpret_cast<float4*>(out.nodes.data());
	for (size_t l = out.level_first.size() - 1; l-- > 0;)
		for (uint32_t i = out.level_first[l]; i < out.level_first[l + 1]; i++) for (int k = 0; k < 4; k++) refit_slot(wide, packed_prims, nullptr, ob, i, k);
	out.ob = ob;
	out.cost = wide_cost(out);
}

void flatten_bvh(const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* prims, uint32_t n_prims, WideBvh& out, const OriginBox* ob_in) {
	out.nodes.clear(); out.prims.clear(); out.max_stack = 0; out.depth = 0; out.tn_bits = 31; out.level_first.assign(1, 0u); out.cost = 0.0;
	sphere_bounds(prims, n_prims, out.sphere_lo, out.sphere_hi);
	const OriginBox ob = ob_in ? *ob_in : origin_box_rule(out.sphere_lo, out.sphere_hi, nullptr, 0);
	out.ob = ob;
	// topology first (links only); the boxes are filled afterwards by the refit routine, deepest level first
	auto set_empty = [](WideNode& w, int k) { for (int j = 0; j < 8; j++) w.slot[k][j] = 0.0f; w.slot[k][4] = w.slot[k][5] = w.slot[k][7] = -1.0e30f; w.slot[k][6] = int_as_float(kEmptyLink); };
	auto set_link = [&](WideNode& w, int k, int32_t link) { for (int j = 0; j < 8; j++) w.slot[k][j] = 0.0f; w.slot[k][6] = int_as_float(link); };
	auto fill_boxes = [&]() {
		out.prims.resize(n_prims);
		for (uint32_t i = 0; i < n_prims; i++) out.prims[i] = make_float4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq);
		wide_fill_boxes(out, out.prims.data(), ob);
	};
	if (n_prims == 0 || n_nodes == 0) {
		WideNode w; for (int k = 0; k < 4; k++) set_empty(w, k);
		out.nodes.push_back(w); out.level_first.push_back(1u); return;
	}
	if (nodes[0].prim_count != 0) {  // single sphere: the root is a leaf
		WideNode w; for (int k = 0; k < 4; k++) set_empty(w, k);
		set_link(w, 0, ~static_cast<int32_t>(nodes[0].first_id));
		out.nodes.push_back(w); out.level_first.push_back(1u); out.depth = 1; fill_boxes(); return;
	}
	// breadth-first: queue entries are binary inner nodes that become wide nodes
	struct Pending { uint32_t bin; uint32_t level; };
	std::vector<Pending> queue; queue.push_back({0u, 1u});
	std::vector<uint32_t> inner_children;   // per wide node: how many of its slots are inner (for the stack bound)
	out.nodes.reserve(n_nodes / 2 + 1);
	for (size_t head = 0; head < queue.size(); head++) {
		const Pending cur = queue[head];
		if (cur.level > out.depth) { out.depth = cur.level; if (cur.level > 1) out.level_first.push_back(static_cast<uint32_t>(head)); }  // first node of a new BFS level
		uint32_t kids[4]; int nk = 2;
		kids[0] = nodes[cur.bin].first_id; kids[1] = kids[0] + 1;
		while (nk < 4) {  // open the inner child with the largest surface until four slots are used
			int pick = -1; float best = -1.0f;
			for (int k = 0; k < nk; k++) if (nodes[kids[k]].prim_count == 0) { const float a = surface(nodes[kids[k]]); if (a > best) { best = a; pick = k; } }
			if (pick < 0) break;
			const uint32_t open = kids[pick];
			kids[pick] = nodes[open].first_id; kids[nk++] = nodes[open].first_id + 1;
		}
		// slot order: inner children first, then leaves
		std::stable_sort(kids, kids + nk, [&](uint32_t x, uint32_t y) { return (nodes[x].prim_count == 0) > (nodes[y].prim_count == 0); });
		WideNode w; uint32_t n_inner = 0;
		for (int k = 0; k < 4; k++) {
			if (k >= nk) { set_empty(w, k); continue; }
			const b2r_bvh_node& c = nodes[kids[k]];
			if (c.prim_count != 0) { set_link(w, k, ~static_cast<int32_t>(c.first_id)); continue; }
			set_link(w, k, static_cast<int32_t>(queue.size()));  // its wide index = its queue position
			queue.push_back({kids[k], cur.level + 1});
			n_inner++;
		}
		out.nodes.push_back(w);
		inner_children.push_back(n_inner);
	}
	// worst-case stack: going into one inner child leaves (inner-1) siblings pushed. Children have larger indices (BFS),
	// so one reverse pass computes need[node] = max over inner children (inner-1 + need[child]).
	std::vector<uint32_t> need(out.nodes.size(), 0);
	for (size_t i = out.nodes.size(); i-- > 0;) {
		uint32_t worst = 0;
		for (int k = 0; k < 4; k++) {
			int32_t link; std::memcpy(&link, &out.nodes[i].slot[k][6], 4);
			if (link >= 0) worst = std::max(worst, inner_children[i] - 1 + need[static_cast<size_t>(link)]);
		}
		need[i] = worst;
	}
	out.max_stack = need[0];
	out.level_first.push_back(static_cast<uint32_t>(out.nodes.size()));
	fill_boxes();
	uint32_t node_bits = 1; while ((1ull << node_bits) < out.nodes.size()) node_bits++;
	out.tn_bits = std::min(32u - node_bits, 29u);  // >= 2 low key bits are dropped: the kernels keep the slot index there
}

void morton_keys(const b2r_sphere* prims, uint32_t n, const float lo[3], const float hi[3], std::vector<uint32_t>& keys) {
	float scale[3]; morton_scale(lo, hi, scale);
	keys.resize(n);
	for (uint32_t i = 0; i < n; i++) keys[i] = morton_key(prims[i].position[0], prims[i].position[1], prims[i].position[2], lo, scale);
}
void packed_levels(uint32_t n, std::vector<uint32_t>& level_first) {
	std::vector<uint32_t> sizes;  // bottom level first
	uint32_t m = (n + 3u) / 4u; if (m == 0u) m = 1u;
	sizes.push_back(m);
	while (m > 1u) { m = (m + 3u) / 4u; sizes.push_back(m); }
	level_first.assign(1, 0u);
	for (size_t l = sizes.size(); l-- > 0;) level_first.push_back(level_first.back() + sizes[l]);
}
void build_packed_tree(const b2r_sphere* prims, uint32_t n, WideBvh& out, const OriginBox* ob_in) {
	out.nodes.clear(); out.prims.clear(); out.geom_of_prim.clear(); out.cost = 0.0;
	sphere_bounds(prims, n, out.sphere_lo, out.sphere_hi);
	const OriginBox ob = ob_in ? *ob_in : origin_box_rule(out.sphere_lo, out.sphere_hi, nullptr, 0);
	std::vector<uint32_t> keys; morton_keys(prims, n, out.sphere_lo, out.sphere_hi, keys);
	std::vector<uint32_t> order(n); std::iota(order.begin(), order.end(), 0u);
	std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });  // == a stable radix sort by key
	packed_levels(n, out.level_first);
	const uint32_t levels = static_cast<uint32_t>(out.level_first.size()) - 1u;
	out.depth = levels; out.max_stack = 3u * levels;
	out.nodes.resize(out.level_first.back());
	for (uint32_t l = 0; l < levels; l++) {
		const uint32_t first = out.level_first[l], count = out.level_first[l + 1] - first;
		const bool bottom = l + 1 == levels;
		const uint32_t child_first = bottom ? 0u : out.level_first[l + 1], child_count = bottom ? n : out.level_first[l + 2] - out.level_first[l + 1];
		for (uint32_t i = 0; i < count; i++) for (int k = 0; k < 4; k++) {
			WideNode& w = out.nodes[first + i];
			for (int j = 0; j < 8; j++) w.slot[k][j] = 0.0f;
			const uint32_t c = 4u * i + static_cast<uint32_t>(k);
			if (c >= child_count) { w.slot[k][4] = w.slot[k][5] = w.slot[k][7] = -1.0e30f; w.slot[k][6] = int_as_float(kEmptyLink); }
			else w.slot[k][6] = int_as_float(bottom ? ~static_cast<int32_t>(order[c]) : static_cast<int32_t>(child_first + c));
		}
	}
	out.prims.resize(n);
	for (uint32_t i = 0; i < n; i++) out.prims[i] = make_float4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq);
	wide_fill_boxes(out, out.prims.data(), ob);
	uint32_t node_bits = 1; while ((1ull << node_bits) < out.nodes.size()) node_bits++;
	out.tn_bits = std::min(32u - node_bits, 29u);
}

bool build_sweep_tree(const b2r_sphere* prims, uint32_t n, WideBvh& out, const OriginBox* ob_in) {
	if (n < 2u) { build_packed_tree(prims, n, out, ob_in); return true; }
	out.nodes.clear(); out.prims.clear(); out.geom_of_prim.clear(); out.cost = 0.0;
	sphere_bounds(prims, n, out.sphere_lo, out.sphere_hi);
	const OriginBox ob = ob_in ? *ob_in : origin_box_rule(out.sphere_lo, out.sphere_hi, nullptr, 0);
	std::vector<uint32_t> keys; morton_keys(prims, n, out.sphere_lo, out.sphere_hi, keys);
	std::vector<uint32_t> order(n); std::iota(order.begin(), order.end(), 0u);
	std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
	std::vector<SweepItem> box(n);
	for (uint32_t p = 0; p < n; p++) { const b2r_sphere& sp = prims[order[p]]; sweep_sphere_box(make_float4(sp.position[0], sp.position[1], sp.position[2], sp.radius_sq), &box[p]); }
	// what the device works out for every run with two segmented scans and an atomic minimum, here one run at a time: the cheapest cut
	// and the area of the run's box, both filed under the run's first position
	std::vector<unsigned long long> cut_of(n, ~0ull); std::vector<float> area_of(n, 0.0f); std::vector<SweepItem> suffix;
	auto survey = [&](uint32_t a, uint32_t b) {
		if (b - a < 2u) return;
		suffix.resize(b - a);
		SweepItem acc = box[b - 1]; acc.flag = 0u; suffix[b - 1 - a] = acc;
		for (uint32_t p = b - 1; p-- > a;) { SweepItem it = box[p]; it.flag = 0u; acc = sweep_join(it, acc); suffix[p - a] = acc; }
		unsigned long long best = ~0ull;
		acc = box[a]; acc.flag = 0u;
		for (uint32_t p = a + 1; p < b; p++) {
			const unsigned long long key = sweep_key(sweep_area(acc), p - a, sweep_area(suffix[p - a]), b - p, p);
			if (key < best) best = key;
			SweepItem it = box[p]; it.flag = 0u; acc = sweep_join(acc, it);
		}
		cut_of[a] = best; area_of[a] = sweep_area(acc);
	};
	struct Run { uint32_t a, b; };
	std::vector<Run> cur(1, Run{0u, n}), next;
	out.level_first.assign(1, 0u);
	auto set_link = [](WideNode& w, int k, int32_t link) {
		for (int j = 0; j < 8; j++) w.slot[k][j] = 0.0f;
		if (link == kEmptyLink) w.slot[k][4] = w.slot[k][5] = w.slot[k][7] = -1.0e30f;
		w.slot[k][6] = int_as_float(link);
	};
	while (!cur.empty()) {
		if (out.level_first.size() > kSweepMaxLevels) return false;  // deeper than the traversal stack allows: the caller builds the packed tree instead
		const uint32_t child_level_first = out.level_first.back() + static_cast<uint32_t>(cur.size());
		out.level_first.push_back(child_level_first);
		next.clear();
		for (const Run& r : cur) {
			SweepKids K{}; K.a[0] = r.a; K.b[0] = r.b; K.n = 1u;
			survey(r.a, r.b);
			for (int round = 0; round < 3; round++) {
				if (!sweep_open(K, cut_of.data(), area_of.data())) break;
				// the two runs the cut made are surveyed for the next round (the device re-surveys every run of the array every round)
				const uint32_t right = K.n - 1u;
				survey(K.a[right], K.b[right]);
				for (uint32_t k = 0; k < right; k++) if (K.b[k] == K.a[right]) survey(K.a[k], K.b[k]);  // the shortened left part
			}
			int32_t link[4]; uint32_t ca[4], cb[4];
			const uint32_t ni = sweep_links(K, order.data(), child_level_first + static_cast<uint32_t>(next.size()), link, ca, cb);
			for (uint32_t i = 0; i < ni; i++) next.push_back(Run{ca[i], cb[i]});
			WideNode w; for (int k = 0; k < 4; k++) set_link(w, k, link[k]);
			out.nodes.push_back(w);
		}
		cur.swap(next);
	}
	const uint32_t levels = static_cast<uint32_t>(out.level_first.size()) - 1u;
	out.depth = levels; out.max_stack = 3u * levels;
	out.prims.resize(n);
	for (uint32_t i = 0; i < n; i++) out.prims[i] = make_float4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq);
	wide_fill_boxes(out, out.prims.data(), ob);
	uint32_t node_bits = 1; while ((1ull << node_bits) < out.nodes.size()) node_bits++;
	out.tn_bits = std::min(32u - node_bits, 29u);
	return true;
}

bool build_sweep3_tree(const b2r_sphere* prims, uint32_t n, WideBvh& out, const OriginBox* ob_in) {
	if (n < 2u) { build_packed_tree(prims, n, out, ob_in); return true; }
	out.nodes.clear(); out.prims.clear(); out.geom_of_prim.clear(); out.cost = 0.0;
	sphere_bounds(prims, n, out.sphere_lo, out.sphere_hi);
	const OriginBox ob = ob_in ? *ob_in : origin_box_rule(out.sphere_lo, out.sphere_hi, nullptr, 0);
	std::vector<SweepItem> box(n);   // by sphere index
	for (uint32_t i = 0; i < n; i++) sweep_sphere_box(make_float4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq), &box[i]);
	std::vector<uint32_t> ord[3], tmp(n); std::vector<unsigned char> right(n, 0);
	for (int ax = 0; ax < 3; ax++) {
		ord[ax].resize(n); std::iota(ord[ax].begin(), ord[ax].end(), 0u);
		std::stable_sort(ord[ax].begin(), ord[ax].end(), [&](uint32_t a, uint32_t b) { return float_order_key(prims[a].position[ax]) < float_order_key(prims[b].position[ax]); });  // == a stable radix sort by key
	}
	std::vector<unsigned long long> cut_of(n, ~0ull); std::vector<float> area_of(n, 0.0f); std::vector<SweepItem> suffix;
	auto survey = [&](uint32_t a, uint32_t b) {
		if (b - a < 2u) return;
		suffix.resize(b - a);
		unsigned long long best = ~0ull; SweepItem acc;
		for (uint32_t ax = 0; ax < 3u; ax++) {
			const uint32_t* o = ord[ax].data();
			acc = box[o[b - 1]]; acc.flag = 0u; suffix[b - 1 - a] = acc;
			for (uint32_t p = b - 1; p-- > a;) { SweepItem it = box[o[p]]; it.flag = 0u; acc = sweep_join(it, acc); suffix[p - a] = acc; }
			acc = box[o[a]]; acc.flag = 0u;
			for (uint32_t p = a + 1; p < b; p++) {
				const unsigned long long key = sweep_key3(sweep_area(acc), p - a, sweep_area(suffix[p - a]), b - p, p, ax);
				if (key < best) best = key;
				SweepItem it = box[o[p]]; it.flag = 0u; acc = sweep_join(acc, it);
			}
		}
		cut_of[a] = best; area_of[a] = sweep_area(acc);
	};
	struct Run { uint32_t a, b; };
	std::vector<Run> cur(1, Run{0u, n}), next;
	out.level_first.assign(1, 0u);
	auto set_link = [](WideNode& w, int k, int32_t link) {
		for (int j = 0; j < 8; j++) w.slot[k][j] = 0.0f;
		if (link == kEmptyLink) w.slot[k][4] = w.slot[k][5] = w.slot[k][7] = -1.0e30f;
		w.slot[k][6] = int_as_float(link);
	};
	while (!cur.empty()) {
		if (out.level_first.size() > kSweepMaxLevels) return false;
		const uint32_t child_level_first = out.level_first.back() + static_cast<uint32_t>(cur.size());
		out.level_first.push_back(child_level_first);
		next.clear();
		for (const Run& r : cur) {
			SweepKids K{}; K.a[0] = r.a; K.b[0] = r.b; K.n = 1u;
			survey(r.a, r.b);
			for (int round = 0; round < 3; round++) {
				uint32_t ax = 0, a = 0, b = 0;
				const uint32_t pos = sweep_open3(K, cut_of.data(), area_of.data(), &ax, &a, &b);
				if (!pos) break;
				// the cut run [a, b): the first pos - a spheres of the chosen axis' order go left; the other two orders are partitioned to match, stably
				for (uint32_t p = a; p < b; p++) right[ord[ax][p]] = p >= pos ? 1 : 0;
				for (uint32_t a2 = 0; a2 < 3u; a2++) {
					if (a2 == ax) continue;
					uint32_t l = a, rr = pos;
					for (uint32_t p = a; p < b; p++) { const uint32_t id = ord[a2][p]; if (right[id]) tmp[rr++] = id; else tmp[l++] = id; }
					std::copy(tmp.begin() + a, tmp.begin() + b, ord[a2].begin() + a);
				}
				survey(a, pos); survey(pos, b);
			}
			int32_t link[4]; uint32_t ca[4], cb[4];
			const uint32_t ni = sweep_links(K, ord[0].data(), child_level_first + static_cast<uint32_t>(next.size()), link, ca, cb);
			for (uint32_t i = 0; i < ni; i++) next.push_back(Run{ca[i], cb[i]});
			WideNode w; for (int k = 0; k < 4; k++) set_link(w, k, link[k]);
			out.nodes.push_back(w);
		}
		cur.swap(next);
	}
	const uint32_t levels = static_cast<uint32_t>(out.level_first.size()) - 1u;
	out.depth = levels; out.max_stack = 3u * levels;
	out.prims.resize(n);
	for (uint32_t i = 0; i < n; i++) out.prims[i] = make_float4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq);
	wide_fill_boxes(out, out.prims.data(), ob);
	uint32_t node_bits = 1; while ((1ull << node_bits) < out.nodes.size()) node_bits++;
	out.tn_bits = std::min(32u - node_bits, 29u);
	return true;
}

void pack_scene(const b2r_sphere* prims, uint32_t n_prims, const b2r_material* materials, uint32_t n_mat,
                const int32_t* light_geom_idx, uint32_t n_lights, const b2r_sphere* geometry, PackedScene& out) {
	auto f4 = [](float x, float y, float z, float w) { float4 v; v.x = x; v.y = y; v.z = z; v.w = w; return v; };
	out.prims.resize(n_prims); out.prim_mat.resize(n_prims);
	for (uint32_t i = 0; i < n_prims; i++) {
		out.prims[i] = f4(prims[i].position[0], prims[i].position[1], prims[i].position[2], prims[i].radius_sq);
		out.prim_mat[i] = prims[i].material_ID;
	}
	out.mat_albedo.resize(n_mat); out.mat_emission.resize(n_mat); out.mat_f0.resize(n_mat); out.mat_diel.resize(n_mat);
	for (uint32_t i = 0; i < n_mat; i++) {
		const float* e = materials[i].emission;
		const bool emissive = sel_max(e[0], sel_max(e[1], e[2])) > FLT_EPSILON;  // is_emissive, Renderer.hpp:201
		out.mat_albedo[i] = f4(materials[i].albedo[0], materials[i].albedo[1], materials[i].albedo[2], emissive ? 1.0f : 0.0f);
		out.mat_emission[i] = f4(e[0], e[1], e[2], 0.0f);
		out.mat_f0[i] = f4(materials[i].F0[0], materials[i].F0[1], materials[i].F0[2], materials[i].roughness);  // Closure<GGX>, Renderer.hpp:210-211
		const float* t = materials[i].transmission;
		const bool diel = sel_max(t[0], sel_max(t[1], t[2])) > 0.0f;  // B2R_FLAG_DIELECTRIC: eta = 0 marks a material that is not dielectric
		out.mat_diel[i] = diel ? f4(t[0], t[1], t[2], 1.0f + materials[i].IOR_minus_one) : f4(0.0f, 0.0f, 0.0f, 0.0f);
	}
	out.light_sphere.resize(n_lights ? n_lights : 1, f4(0, 0, 0, 0)); out.light_emit.resize(n_lights ? n_lights : 1, f4(0, 0, 0, 0));
	for (uint32_t i = 0; i < n_lights; i++) {  // NEE reads the light from scene.geometry, original order (Renderer.hpp:261-262,277)
		const b2r_sphere& g = geometry[light_geom_idx[i]];
		const float* e = materials[g.material_ID].emission;
		out.light_sphere[i] = f4(g.position[0], g.position[1], g.position[2], g.radius_sq);
		out.light_emit[i] = f4(e[0], e[1], e[2], int_as_float(light_geom_idx[i]));
	}
}

bool dielectric_materials_valid(const b2r_material* materials, uint32_t n_mat) {
	for (uint32_t i = 0; i < n_mat; i++) {
		const float* t = materials[i].transmission;
		if (!std::isfinite(t[0]) || !std::isfinite(t[1]) || !std::isfinite(t[2])) return false;
		if (!(sel_max(t[0], sel_max(t[1], t[2])) > 0.0f)) continue;
		const float eta = 1.0f + materials[i].IOR_minus_one;
		for (int k = 0; k < 3; k++) if (!(t[k] >= 0.0f && t[k] <= 1.0f)) return false;
		if (!std::isfinite(eta) || !(eta >= 1.0f)) return false;
	}
	return true;
}

}  // namespace b2r

// ---------------------------------------------------------------------------------------------- C ABI (host-only part)
extern "C" {

int b2r_bvh_build(const b2r_sphere* geometry, uint32_t n, b2r_bvh_node* nodes_out, b2r_sphere* prims_out,
                  uint32_t* prim_ids_out, uint32_t* n_nodes_out) {
	return b2r_bvh_build_ex(geometry, n, 0u, 1.0f, nodes_out, prims_out, prim_ids_out, n_nodes_out);
}

int b2r_bvh_build_ex(const b2r_sphere* geometry, uint32_t n, uint32_t log_cluster_size, float cost_ratio, b2r_bvh_node* nodes_out,
                     b2r_sphere* prims_out, uint32_t* prim_ids_out, uint32_t* n_nodes_out) {
	if ((n && !geometry) || !nodes_out || log_cluster_size > 31u) return B2R_ERR_ARG;
	std::vector<b2r_bvh_node> nodes; std::vector<b2r_sphere> prims; std::vector<uint32_t> ids;
	b2r::build_reference_bvh(geometry, n, nodes, prims, ids, log_cluster_size, cost_ratio);
	std::memcpy(nodes_out, nodes.data(), nodes.size() * sizeof(b2r_bvh_node));
	if (prims_out && n) std::memcpy(prims_out, prims.data(), prims.size() * sizeof(b2r_sphere));
	if (prim_ids_out && n) std::memcpy(prim_ids_out, ids.data(), ids.size() * sizeof(uint32_t));
	if (n_nodes_out) *n_nodes_out = static_cast<uint32_t>(nodes.size());
	return B2R_OK;
}

int b2r_find_lights(const b2r_sphere* geometry, uint32_t n, const b2r_material* materials, uint32_t n_mat,
                    int32_t* out, uint32_t* n_out) {
	if ((n && !geometry) || (n && !materials) || !n_out) return B2R_ERR_ARG;
	uint32_t count = 0;
	for (uint32_t i = 0; i < n; i++) {  // Scene.hpp:12-16: dot(emission, emission) > 0
		const int32_t m = geometry[i].material_ID;
		if (m < 0 || static_cast<uint32_t>(m) >= n_mat) return B2R_ERR_ARG;
		const float* e = materials[m].emission;
		if (e[0] * e[0] + e[1] * e[1] + e[2] * e[2] > 0.0f) { if (out) out[count] = static_cast<int32_t>(i); count++; }
	}
	*n_out = count;
	return B2R_OK;
}

int b2r_camera_ray(const float pos[3], const float q[4], float half_width, float half_height, float z, int32_t x, int32_t y, const float samples[2], float origin_out[3], float dir_out[3]) {
	if (!pos || !q || !samples || !origin_out || !dir_out) return B2R_ERR_ARG;
	const b2r::CameraParams cam{pos[0], pos[1], pos[2], q[0], q[1], q[2], q[3], half_width, half_height, z, 1.0f};
	const b2r::f3 d = b2r::camera_dir(cam, x, y, samples[0], samples[1]);  // the routine the kernels run per pixel (b2r_math.h)
	origin_out[0] = pos[0]; origin_out[1] = pos[1]; origin_out[2] = pos[2];
	dir_out[0] = d.x; dir_out[1] = d.y; dir_out[2] = d.z;
	return B2R_OK;
}

int b2r_camera_lookat(const float eye[3], const float dir[3], uint32_t width, uint32_t height, float focal_length_mm,
                      float exposure, float out11[11]) {
	if (!eye || !dir || !out11) return B2R_ERR_ARG;
	out11[0] = eye[0]; out11[1] = eye[1]; out11[2] = eye[2];
	b2r::look_at_quat(b2r::f3{dir[0], dir[1], dir[2]}, out11 + 3);
	const float inv_half_tan = (-2.0f / 24.0f) * focal_length_mm;  // Projection::UpdateLens, Camera.hpp:21-26 (24 mm sensor)
	out11[7] = static_cast<float>(width) * 0.5f;                   // Projection::Resize, Camera.hpp:28-32
	out11[8] = static_cast<float>(height) * 0.5f;
	out11[9] = out11[8] * inv_half_tan;
	out11[10] = exposure;
	return B2R_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------- traversal tree
// The reference's tree (above) must keep its node order, quirks included: its split "area" is only extent.y*extent.z (Q17),
// which yields long, overlapping boxes — about 46 wide-node visits and 58 sphere tests per primary ray on the 100k-sphere
// scene. Traversal results do not depend on the tree (closest hit == brute force over all spheres; leaf links carry the
// reference's leaf index), so the GPU walks a tree built for traversal instead: binned SAH over the true surface area,
// one sphere per leaf, emitted in the same {box, first_id, prim_count} node format so flatten_bvh() is shared.
namespace b2r {
namespace {
struct TBox { float lo[3], hi[3]; };
inline TBox tbox_empty() { return TBox{{FLT_MAX, FLT_MAX, FLT_MAX}, {-FLT_MAX, -FLT_MAX, -FLT_MAX}}; }
inline void tbox_grow(TBox& a, const TBox& b) { for (int k = 0; k < 3; k++) { a.lo[k] = fminf(a.lo[k], b.lo[k]); a.hi[k] = fmaxf(a.hi[k], b.hi[k]); } }
inline float tbox_area(const TBox& b) { const float x = b.hi[0] - b.lo[0], y = b.hi[1] - b.lo[1], z = b.hi[2] - b.lo[2]; return x * y + y * z + z * x; }
}  // namespace

namespace {
// One subtree of the traversal tree. Node indices are fixed by the subtree sizes alone — the children of a node sit next to each
// other at `region`, followed by all descendants of the left child (2*left - 2 nodes) and then those of the right one — so
// subtrees can be built by different threads into the pre-sized node array and the result does not depend on the schedule.
struct TraversalBuilder {
	static constexpr int kBins = 16;
	const std::vector<TBox>& box; const std::vector<float>& cen; std::vector<uint32_t>& ids; std::vector<b2r_bvh_node>& nodes;
	void set(uint32_t node, const TBox& b, uint32_t first, uint32_t count) {
		b2r_bvh_node nd; for (int k = 0; k < 3; k++) { nd.min_bound[k] = b.lo[k]; nd.max_bound[k] = b.hi[k]; } nd.first_id = first; nd.prim_count = count; nodes[node] = nd;
	}
	// runs fn(chunk, b, e) over `workers` equal chunks of [begin, end), chunk 0 on the calling thread
	template <class F> static void chunks(uint32_t begin, uint32_t end, unsigned workers, F&& fn) {
		const uint32_t count = end - begin, step = (count + workers - 1) / workers;
		std::vector<std::thread> pool;
		for (unsigned w = 1; w < workers; w++) { const uint32_t b = begin + std::min(count, w * step), e = begin + std::min(count, (w + 1) * step); if (b < e) pool.emplace_back([&fn, w, b, e] { fn(w, b, e); }); }
		fn(0u, begin, begin + std::min(count, step));
		for (auto& t : pool) t.join();
	}
	struct Bins { TBox bb[3][kBins]; uint32_t bc[3][kBins]; };
	// splits [begin, end) of node `node`; returns the split position and writes the two children at `region`. `workers` > 1: the
	// passes over a large node (the top of the tree is the serial part of the build) are shared out in chunks; every quantity merged
	// across chunks is a min, a max or an integer count, and the degenerate split is made on sorted ids, so the tree is a function of
	// the SET of spheres in the node — not of their order, of the partition algorithm or of the number of threads.
	uint32_t split(uint32_t node, uint32_t begin, uint32_t end, uint32_t region, unsigned workers) {
		const uint32_t count = end - begin;
		if (count < 32768u) workers = 1;
		float clo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, chi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
		{
			std::vector<std::array<float, 6>> part(workers, std::array<float, 6>{FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX});
			chunks(begin, end, workers, [&](unsigned w, uint32_t b, uint32_t e) {
				std::array<float, 6> a = part[w];
				for (uint32_t i = b; i < e; i++) for (int k = 0; k < 3; k++) { const float c = cen[3 * static_cast<size_t>(ids[i]) + k]; a[k] = fminf(a[k], c); a[3 + k] = fmaxf(a[3 + k], c); }
				part[w] = a; });
			for (const auto& a : part) for (int k = 0; k < 3; k++) { clo[k] = fminf(clo[k], a[k]); chi[k] = fmaxf(chi[k], a[3 + k]); }
		}
		// binned SAH: one pass fills the bins of all three axes
		float scale[3]; bool usable[3];
		for (int axis = 0; axis < 3; axis++) { const float ext = chi[axis] - clo[axis]; usable[axis] = ext > 0.0f; scale[axis] = usable[axis] ? kBins / ext : 0.0f; }
		std::vector<Bins> bins(workers);
		chunks(begin, end, workers, [&](unsigned w, uint32_t b, uint32_t e) {
			Bins& bn = bins[w];
			for (int axis = 0; axis < 3; axis++) for (int q = 0; q < kBins; q++) { bn.bb[axis][q] = tbox_empty(); bn.bc[axis][q] = 0; }
			for (uint32_t i = b; i < e; i++) {
				const uint32_t id = ids[i]; const TBox& bx = box[id];
				for (int axis = 0; axis < 3; axis++) {
					if (!usable[axis]) continue;
					int q = static_cast<int>((cen[3 * static_cast<size_t>(id) + axis] - clo[axis]) * scale[axis]); if (q >= kBins) q = kBins - 1;
					tbox_grow(bn.bb[axis][q], bx); bn.bc[axis][q]++;
				}
			} });
		Bins& all = bins[0];
		for (unsigned w = 1; w < workers; w++) for (int axis = 0; axis < 3; axis++) for (int q = 0; q < kBins; q++) { tbox_grow(all.bb[axis][q], bins[w].bb[axis][q]); all.bc[axis][q] += bins[w].bc[axis][q]; }
		int best_axis = -1, best_bin = 0; float best_cost = FLT_MAX;
		for (int axis = 0; axis < 3; axis++) {  // first axis wins ties
			if (!usable[axis]) continue;
			const TBox* bb = all.bb[axis]; const uint32_t* bc = all.bc[axis];
			float right_area[kBins]; uint32_t right_cnt[kBins];
			TBox acc = tbox_empty(); uint32_t cnt = 0;
			for (int q = kBins - 1; q > 0; q--) { tbox_grow(acc, bb[q]); cnt += bc[q]; right_area[q] = cnt ? tbox_area(acc) : 0.0f; right_cnt[q] = cnt; }
			acc = tbox_empty(); cnt = 0;
			for (int q = 0; q + 1 < kBins; q++) {
				tbox_grow(acc, bb[q]); cnt += bc[q];
				if (cnt == 0 || right_cnt[q + 1] == 0) continue;
				const float cost = tbox_area(acc) * cnt + right_area[q + 1] * right_cnt[q + 1];
				if (cost < best_cost) { best_cost = cost; best_axis = axis; best_bin = q; }
			}
		}
		uint32_t mid = begin;
		if (best_axis >= 0) {
			const float sc = scale[best_axis], lo = clo[best_axis];
			auto goes_left = [&](uint32_t id) { int q = static_cast<int>((cen[3 * static_cast<size_t>(id) + best_axis] - lo) * sc); if (q >= kBins) q = kBins - 1; return q <= best_bin; };
			if (workers == 1) mid = static_cast<uint32_t>(std::partition(ids.begin() + begin, ids.begin() + end, goes_left) - ids.begin());
			else {  // chunk-wise partition into a scratch copy: left parts, then right parts, in chunk order
				std::vector<uint32_t> scratch(ids.begin() + begin, ids.begin() + end), n_left(workers, 0u), first(workers, 0u), last(workers, 0u);
				chunks(begin, end, workers, [&](unsigned w, uint32_t b, uint32_t e) { uint32_t c = 0; for (uint32_t i = b; i < e; i++) c += goes_left(scratch[i - begin]) ? 1u : 0u; n_left[w] = c; first[w] = b; last[w] = e; });
				uint32_t total_left = 0; for (unsigned w = 0; w < workers; w++) total_left += n_left[w];
				std::vector<uint32_t> at_left(workers), at_right(workers);
				uint32_t l = begin, r = begin + total_left;
				for (unsigned w = 0; w < workers; w++) { at_left[w] = l; at_right[w] = r; l += n_left[w]; r += (last[w] - first[w]) - n_left[w]; }
				chunks(begin, end, workers, [&](unsigned w, uint32_t b, uint32_t e) { uint32_t l2 = at_left[w], r2 = at_right[w]; for (uint32_t i = b; i < e; i++) { const uint32_t id = scratch[i - begin]; if (goes_left(id)) ids[l2++] = id; else ids[r2++] = id; } });
				mid = begin + total_left;
			}
		}
		TBox l = tbox_empty(), r = tbox_empty();
		if (best_axis < 0 || mid == begin || mid == end) {  // all centroids coincide: halve the list, on sorted ids so that the result does not depend on the order
			std::sort(ids.begin() + begin, ids.begin() + end);
			mid = begin + count / 2;
			for (uint32_t i = begin; i < mid; i++) tbox_grow(l, box[ids[i]]);
			for (uint32_t i = mid; i < end; i++) tbox_grow(r, box[ids[i]]);
		} else {  // the children's boxes are the unions of the bins on either side of the split (the same min / max over the same boxes)
			for (int q = 0; q <= best_bin; q++) tbox_grow(l, all.bb[best_axis][q]);
			for (int q = best_bin + 1; q < kBins; q++) tbox_grow(r, all.bb[best_axis][q]);
		}
		set(region, l, 0, 0); set(region + 1, r, 0, 0);
		nodes[node].first_id = region; nodes[node].prim_count = 0;
		return mid;
	}
	struct Job { uint32_t node, begin, end, region; };
	void build(Job root, std::vector<Job>* spill, uint32_t spill_above, unsigned workers) {
		std::vector<Job> todo; todo.push_back(root);
		while (!todo.empty()) {
			const Job j = todo.back(); todo.pop_back();
			const uint32_t count = j.end - j.begin;
			if (count == 1) { nodes[j.node].first_id = ids[j.begin]; nodes[j.node].prim_count = 1; continue; }
			if (spill && count <= spill_above && count > 1 && j.node != root.node) { spill->push_back(j); continue; }  // handed to the thread pool
			const uint32_t mid = split(j.node, j.begin, j.end, j.region, workers);
			const uint32_t left = mid - j.begin;
			todo.push_back({j.region, j.begin, mid, j.region + 2u});
			todo.push_back({j.region + 1u, mid, j.end, j.region + 2u + (2u * left - 2u)});
		}
	}
};
}  // namespace

void build_traversal_tree(const b2r_sphere* prims, uint32_t n, std::vector<b2r_bvh_node>& nodes) {
	nodes.clear();
	if (n == 0) { nodes.push_back(to_node(void_box(), 0, 0)); return; }
	std::vector<TBox> box(n); std::vector<float> cen(3 * static_cast<size_t>(n)); std::vector<uint32_t> ids(n);
	for (uint32_t i = 0; i < n; i++) {
		const float r = sqrtf(prims[i].radius_sq);
		for (int k = 0; k < 3; k++) { box[i].lo[k] = prims[i].position[k] - r; box[i].hi[k] = prims[i].position[k] + r; cen[3 * static_cast<size_t>(i) + k] = prims[i].position[k]; }
		ids[i] = i;
	}
	nodes.resize(2 * static_cast<size_t>(n) - 1);
	TraversalBuilder tb{box, cen, ids, nodes};
	TBox root = tbox_empty(); for (uint32_t i = 0; i < n; i++) tbox_grow(root, box[i]);
	tb.set(0, root, 0, 0);
	const unsigned hw = std::thread::hardware_concurrency();
	const unsigned threads = n < 20000u ? 1u : (hw ? (hw > 32u ? 32u : hw) : 1u);
	if (threads <= 1) { tb.build({0u, 0u, n, 1u}, nullptr, 0, 1u); return; }
	// the top of the tree on this thread until the pieces are small enough to share out, then one piece at a time per worker
	std::vector<TraversalBuilder::Job> pieces;
	tb.build({0u, 0u, n, 1u}, &pieces, n / (threads * 4u) + 1u, threads);
	std::sort(pieces.begin(), pieces.end(), [](const TraversalBuilder::Job& a, const TraversalBuilder::Job& b) { return a.end - a.begin > b.end - b.begin; });
	std::atomic<size_t> next{0};
	auto work = [&] { for (;;) { const size_t k = next.fetch_add(1); if (k >= pieces.size()) break; tb.build(pieces[k], nullptr, 0, 1u); } };
	std::vector<std::thread> pool;
	for (unsigned t = 1; t < threads; t++) pool.emplace_back(work);
	work();
	for (auto& t : pool) t.join();
}
}  // namespace b2r

// ---------------------------------------------------------------------------------------------- frame output
// Image::Store (Image.cpp:71-74): stbi_flip_vertically_on_write(true); stbi_write_hdr(path, w, h, 4, rgba). The file format is
// the published Radiance RGBE format with per-scanline run-length encoding; the mantissa/exponent split follows stb's
// linear_to_rgbe (frexp of the largest channel, truncating conversion). Header as stb writes it: the EXPOSURE line follows FORMAT directly
// and ONE empty line ends the header (stb_image's own reader — b2r_read_hdr below — takes the line after the first empty one as the resolution).
extern "C" int b2r_write_hdr(const char* path, const float* rgba, uint32_t width, uint32_t height) {
	if (!path || !rgba || width == 0 || height == 0) return B2R_ERR_ARG;
	FILE* f = std::fopen(path, "wb");
	if (!f) return B2R_ERR_ARG;
	std::fprintf(f, "#?RADIANCE\n# Written by libb2r\nFORMAT=32-bit_rle_rgbe\nEXPOSURE=          1.0000000000000\n\n-Y %u +X %u\n", height, width);
	std::vector<unsigned char> rgbe(static_cast<size_t>(width) * 4), line;
	for (uint32_t row = 0; row < height; row++) {
		const float* src = rgba + static_cast<size_t>(height - 1 - row) * width * 4;  // vertical flip
		for (uint32_t x = 0; x < width; x++) {
			const float r = src[4 * x], g = src[4 * x + 1], b = src[4 * x + 2];
			const float m = fmaxf(r, fmaxf(g, b));
			unsigned char* o = &rgbe[4 * static_cast<size_t>(x)];
			if (m < 1e-32f) { o[0] = o[1] = o[2] = o[3] = 0; continue; }
			int e; const float n = frexpf(m, &e) * 256.0f / m;
			o[0] = static_cast<unsigned char>(r * n); o[1] = static_cast<unsigned char>(g * n); o[2] = static_cast<unsigned char>(b * n); o[3] = static_cast<unsigned char>(e + 128);
		}
		if (width < 8 || width >= 32768) { std::fwrite(rgbe.data(), 1, rgbe.size(), f); continue; }  // flat scanline
		line.clear(); line.push_back(2); line.push_back(2); line.push_back(static_cast<unsigned char>(width >> 8)); line.push_back(static_cast<unsigned char>(width & 255));
		for (int c = 0; c < 4; c++) {  // each component separately, with stb_image_write's own choice of runs and literals (stbiw__write_hdr_scanline)
			uint32_t x = 0;
			auto at = [&](uint32_t k) { return rgbe[4 * static_cast<size_t>(k) + c]; };
			while (x < width) {
				uint32_t r = x;  // the first position where three equal bytes start
				while (r + 2 < width) { if (at(r) == at(r + 1) && at(r) == at(r + 2)) break; ++r; }
				if (r + 2 >= width) r = width;
				while (x < r) {  // literals up to there, at most 128 at a time
					uint32_t len = r - x; if (len > 128) len = 128;
					line.push_back(static_cast<unsigned char>(len)); for (uint32_t k = 0; k < len; k++) line.push_back(at(x + k));
					x += len;
				}
				if (r + 2 < width) {  // the run, at most 127 at a time (a remainder of one or two is still written as a run)
					while (r < width && at(r) == at(x)) ++r;
					while (x < r) {
						uint32_t len = r - x; if (len > 127) len = 127;
						line.push_back(static_cast<unsigned char>(128 + len)); line.push_back(at(x));
						x += len;
					}
				}
			}
		}
		std::fwrite(line.data(), 1, line.size(), f);
	}
	const bool ok = std::fclose(f) == 0;
	return ok ? B2R_OK : B2R_ERR_ARG;
}

// ---------------------------------------------------------------------------------------------- sky texture input
// The reference loads its environment map with stbi_loadf(path, &w, &h, &channels, 4) (Application.cpp:225-231; also Image.cpp:53-55).
// stb_image.h is a third-party header the reference does not vendor (nothings/stb, no pinned version; the .hdr path has been stable
// through v2.x). This restates its published Radiance decoder — stbi__hdr_load / stbi__hdr_convert — for req_comp = 4:
//   header:  first line "#?RADIANCE" or "#?RGBE"; lines up to the first empty one, one of which must be "FORMAT=32-bit_rle_rgbe";
//            then "-Y <height> +X <width>" (no other orientation is accepted);
//   pixels:  width < 8 or >= 32768: flat RGBE quadruples. Otherwise per scanline {2, 2, width_hi, width_lo} followed by the four
//            components one after the other, each as runs (count > 128: count-128 copies of the next byte) and literals (count bytes);
//            a scanline that does not start with {2, 2, <0x80} switches the rest of the file to flat pixels, the four bytes read so
//            far being pixel 0 and decoding resuming at pixel 1 of row 0 — stb's own comment: "yes, this makes no sense";
//   value:   e == 0 -> 0, else channel = mantissa * 2^(e - 136), no half-bit offset; alpha = 1. Rows in file order (no vertical flip
//            unless stbi_set_flip_vertically_on_load was called, which the reference never does).
namespace {
struct ByteReader {
	FILE* f; bool eof = false;
	int get8() { const int c = std::fgetc(f); if (c == EOF) { eof = true; return 0; } return c; }
	void getn(unsigned char* dst, int n) { for (int i = 0; i < n; i++) dst[i] = static_cast<unsigned char>(get8()); }
	// stbi__hdr_gettoken: one line without its '\n', at most 1023 characters kept, the rest of an over-long line skipped
	std::string token() {
		std::string s; int c = get8();
		while (!eof && c != '\n') {
			s.push_back(static_cast<char>(c));
			if (s.size() == 1023) { while (!eof && get8() != '\n') {} break; }
			c = get8();
		}
		return s;
	}
};
inline void rgbe_to_float4(float* out, const unsigned char* in) {  // stbi__hdr_convert, req_comp 4
	if (in[3] != 0) {
		const float f1 = static_cast<float>(ldexp(1.0f, static_cast<int>(in[3]) - (128 + 8)));
		out[0] = in[0] * f1; out[1] = in[1] * f1; out[2] = in[2] * f1;
	} else out[0] = out[1] = out[2] = 0.0f;
	out[3] = 1.0f;
}
}  // namespace

extern "C" int b2r_read_hdr(const char* path, float* rgba_out, int32_t* width_out, int32_t* height_out) {
	if (!path || !width_out || !height_out) return B2R_ERR_ARG;
	FILE* f = std::fopen(path, "rb");
	if (!f) return B2R_ERR_ARG;
	struct Closer { FILE* f; ~Closer() { std::fclose(f); } } closer{f};
	ByteReader in{f};
	const std::string magic = in.token();
	if (magic != "#?RADIANCE" && magic != "#?RGBE") return B2R_ERR_ARG;               // "not HDR"
	bool valid = false;
	for (;;) { const std::string t = in.token(); if (t.empty()) break; if (t == "FORMAT=32-bit_rle_rgbe") valid = true; }
	if (!valid) return B2R_ERR_ARG;                                                      // "unsupported format"
	const std::string res = in.token();
	if (res.compare(0, 3, "-Y ") != 0) return B2R_ERR_ARG;                               // "unsupported data layout"
	char* p = nullptr; const char* s = res.c_str() + 3;
	const long height = std::strtol(s, &p, 10);
	while (*p == ' ') ++p;
	if (std::strncmp(p, "+X ", 3) != 0) return B2R_ERR_ARG;
	const long width = std::strtol(p + 3, nullptr, 10);
	if (height <= 0 || width <= 0 || height > (1 << 24) || width > (1 << 24)) return B2R_ERR_ARG;   // stb: "too large" above STBI_MAX_DIMENSIONS
	*width_out = static_cast<int32_t>(width); *height_out = static_cast<int32_t>(height);
	if (!rgba_out) return B2R_OK;                                                        // size query
	const size_t W = static_cast<size_t>(width), H = static_cast<size_t>(height);
	size_t i = 0, j = 0;
	bool flat = width < 8 || width >= 32768;
	if (!flat) {
		std::vector<unsigned char> scan(W * 4);
		for (j = 0; j < H && !flat; ++j) {
			const int c1 = in.get8(), c2 = in.get8(); int len = in.get8();
			if (c1 != 2 || c2 != 2 || (len & 0x80)) {
				const unsigned char rgbe[4] = {static_cast<unsigned char>(c1), static_cast<unsigned char>(c2), static_cast<unsigned char>(len), static_cast<unsigned char>(in.get8())};
				rgbe_to_float4(rgba_out, rgbe);
				i = 1; j = 0; flat = true;
				break;
			}
			len = (len << 8) | in.get8();
			if (static_cast<long>(len) != width) return B2R_ERR_ARG;                     // "invalid decoded scanline length"
			for (int k = 0; k < 4; ++k) {
				size_t x = 0;
				while (x < W) {
					const size_t nleft = W - x;
					int count = in.get8();
					if (in.eof) return B2R_ERR_ARG;
					if (count > 128) {
						const unsigned char value = static_cast<unsigned char>(in.get8()); count -= 128;
						if (count == 0 || static_cast<size_t>(count) > nleft) return B2R_ERR_ARG;  // "corrupt"
						for (int z = 0; z < count; ++z) scan[x++ * 4 + k] = value;
					} else {
						if (count == 0 || static_cast<size_t>(count) > nleft) return B2R_ERR_ARG;
						for (int z = 0; z < count; ++z) scan[x++ * 4 + k] = static_cast<unsigned char>(in.get8());
					}
				}
			}
			for (size_t x = 0; x < W; ++x) rgbe_to_float4(rgba_out + (j * W + x) * 4, scan.data() + x * 4);
		}
	}
	if (flat) {
		for (; j < H; ++j, i = 0) for (; i < W; ++i) { unsigned char rgbe[4]; in.getn(rgbe, 4); rgbe_to_float4(rgba_out + (j * W + i) * 4, rgbe); }
	}
	return in.eof ? B2R_ERR_ARG : B2R_OK;  // (stb does not notice a short file; a truncated environment map is reported here)
}
