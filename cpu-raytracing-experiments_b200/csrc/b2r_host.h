// b2r_host.h — host-side scene preparation shared by the C ABI (b2r.cu): BVH construction with the reference's
// node/leaf order, and its flattening into the 128-byte 4-wide node layout the traversal kernels read.
#pragma once
#include <stdint.h>
#include <vector>
#include <vector_types.h>
#include "../../include/b2r.h"

namespace b2r {

// 128-byte traversal node: four 32-byte child slots, each two float4 — a box as centre + half extents in EVERY slot:
//   inner child : {c.x, c.y, c.z, 0  } {h.x, h.y, link = wide-node index (>= 0), h.z}
//   leaf child  : {c.x, c.y, c.z, r^2} {H,   H,   link = ~prim_index      (< 0),  H  }   (sphere inlined: no leaf fetch)
//   empty slot  : link = kEmptyLink, h = -1e30 (its box fails the slab test of every ray that keeps an axis constrained, b2r_shade.h slab_setup)
// A leaf's H is the half extent of a cube around the sphere that contains every ray the float sphere tests can report as a hit
// (leaf_half_extent, b2r_shade.h); inner boxes are the padded union of their child node's slot boxes (refit_child_box), so the one
// uniform slab pass of the traversal kernels is conservative for all four slots. The spheres are the reference's prims (BVH leaf
// order), bit-exact.
struct alignas(128) WideNode { float slot[4][8]; };
static_assert(sizeof(WideNode) == 128, "one node = one 128-byte line");
constexpr int32_t kEmptyLink = INT32_MIN;
constexpr int kTraversalStack = 64;  // entries per thread; upload fails with B2R_ERR_BVH if a tree needs more

struct OriginBox { float lo[3], hi[3]; };
struct WideBvh {
	std::vector<WideNode> nodes;   // nodes[0] = root, breadth-first (top of the tree is contiguous)
	uint32_t max_stack = 0;        // worst-case traversal stack occupancy for this tree
	uint32_t tn_bits = 10;         // low bits of a 32-bit stack entry that carry the entry distance (rest: node index)
	uint32_t depth = 0;
	std::vector<uint32_t> level_first;  // nodes of BFS level l are [level_first[l], level_first[l+1]); children always sit on a deeper level
	double cost = 0.0;             // sum of the inner-slot half areas (what a refit is compared against)
	float sphere_lo[3] = {0, 0, 0}, sphere_hi[3] = {0, 0, 0};  // bounds of the spheres the tree was built over
	OriginBox ob{};                // the origin box the leaf extents were computed for
	std::vector<float4> prims;     // the spheres {c.xyz, r^2} the tree was built over (boxes can be recomputed for another origin box)
	std::vector<uint32_t> geom_of_prim;  // for b2r_refit_scene: geometry index of the sphere each BVH-order leaf index stands for (empty: unknown)
};

// BoundingVolumeHierarchy<Sphere> constructor (BVH.hpp:90-206), bit-identical node and leaf order.
void build_reference_bvh(const b2r_sphere* geometry, uint32_t n, std::vector<b2r_bvh_node>& nodes,
                         std::vector<b2r_sphere>& prims, std::vector<uint32_t>& prim_ids, uint32_t log_cluster_size = 0u, float cost_ratio = 1.0f);
// Checks the invariants the flattening relies on (children adjacent, leaf size 1, indices in range). Returns false if malformed.
bool validate_reference_bvh(const b2r_bvh_node* nodes, uint32_t n_nodes, uint32_t n_prims);
// A second binary tree over the same spheres (reference leaf order kept in the leaf links), built for traversal speed.
void build_traversal_tree(const b2r_sphere* prims_bvh_order, uint32_t n, std::vector<b2r_bvh_node>& nodes);
// Where ray origins may lie (the leaves' inflated extents depend on how far a ray origin can be from a sphere, b2r_shade.h
// leaf_half_extent): the bounds of all spheres, plus `extra` points (camera position, caller-supplied ray origins: [n_extra][3]), each
// side widened by an eighth of the extent + 1 so that small moves of the camera or the spheres keep the box. Deterministic: the host
// twin of the tests calls the same rule.
void sphere_bounds(const b2r_sphere* prims, uint32_t n, float lo[3], float hi[3]);
OriginBox origin_box_rule(const float sphere_lo[3], const float sphere_hi[3], const float* extra, uint32_t n_extra);
bool origin_box_holds(const OriginBox& ob, const float* points, uint32_t n_points);
// Collapse the binary tree 2 -> 4 wide, inline the leaf spheres and compute every slot box bottom-up (the refit routine, level by level).
void flatten_bvh(const b2r_bvh_node* nodes, uint32_t n_nodes, const b2r_sphere* prims, uint32_t n_prims, WideBvh& out, const OriginBox* ob = nullptr);
// The traversal tree the GPU can build by itself (b2r_upload_scene with B2R_FLAG_GPU_TREE; k_morton_keys / k_packed_links in
// b2r_device.cuh): spheres sorted by the 30-bit curve key of their centre (its cell's Hilbert index, b2r_shade.h morton_key; stable), packed four to a bottom node, nodes packed four to
// a parent, level by level up to the root — an implicit, perfectly balanced 4-ary topology whose links follow from the sphere count
// alone; the boxes are then filled by the refit routine. This is its host twin (tests compare the device tree with it bit for bit).
void morton_keys(const b2r_sphere* prims, uint32_t n, const float lo[3], const float hi[3], std::vector<uint32_t>& keys);
void build_packed_tree(const b2r_sphere* prims, uint32_t n, WideBvh& out, const OriginBox* ob = nullptr);
// The better tree the GPU can build by itself (B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH; k_sweep_* in b2r_device.cuh): the spheres stay in curve
// order, and every node is a run of that order cut top-down where the surface-area heuristic is smallest ALONG THE CURVE, opened 2 -> 4 wide
// like flatten_bvh's collapse (b2r_shade.h: sweep_*). Host twin, bit for bit. Returns false (out unusable) when the tree would be deeper
// than kSweepMaxLevels — the caller then builds the packed tree.
bool build_sweep_tree(const b2r_sphere* prims, uint32_t n, WideBvh& out, const OriginBox* ob = nullptr);
// The same with three orders instead of one curve (B2R_FLAG_GPU_SAH3): the spheres sorted by centre x, y and z, every cut the cheapest over all
// three (a full-sweep surface-area-heuristic build, as the classic CPU builders do it), the two other orders partitioned to match. Host twin.
bool build_sweep3_tree(const b2r_sphere* prims, uint32_t n, WideBvh& out, const OriginBox* ob = nullptr);
// level sizes of the packed tree for n spheres, root level first (level_first has one more entry than there are levels)
void packed_levels(uint32_t n, std::vector<uint32_t>& level_first);
// (Re)compute every slot box of a flattened topology for the spheres `prims` and the origin box `ob` (what flatten_bvh ends with).
void wide_fill_boxes(WideBvh& tree, const float4* packed_prims /*{c.xyz, r^2}, BVH leaf order*/, const OriginBox& ob);
// Sum of the inner-slot half areas of a flattened tree (WideBvh::cost; k_tree_cost computes the same sum on the device after a refit).
double wide_cost(const WideBvh& tree);
// prims (BVH leaf order) as a permutation of geometry (original order), matched by value — the reference's BVH keeps reordered COPIES
// of the spheres and no index map (BVH.hpp:201-205). geom_of_prim[i] = index into geometry of prims[i]; equal spheres are paired in
// index order. Returns false when prims is not a permutation of geometry.
bool match_prims_to_geometry(const b2r_sphere* prims, const b2r_sphere* geometry, uint32_t n, std::vector<uint32_t>& geom_of_prim);


// Scene arrays in the packed form the kernels read (SceneDev): spheres {c.xyz, r^2} in BVH leaf order, per-material
// {albedo, emissive flag} and {emission}, per-light {sphere of scene.geometry[light]} and {emission, light_primID}.
struct PackedScene {
	std::vector<float4> prims, mat_albedo, mat_emission, mat_f0, light_sphere, light_emit;
	std::vector<int32_t> prim_mat;
};
void pack_scene(const b2r_sphere* prims, uint32_t n_prims, const b2r_material* materials, uint32_t n_mat,
                const int32_t* light_geom_idx, uint32_t n_lights, const b2r_sphere* geometry, PackedScene& out);

}  // namespace b2r
