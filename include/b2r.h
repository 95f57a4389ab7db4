/* b2r.h — C ABI of the B200-native wavefront path tracer (libb2r.so).
 *
 * Drop-in boundary for ONE hot path of Borx25/CPU-Raytracing-experiments: Renderer::Accumulate
 * (Renderer.hpp:73-434), Renderer::Render (Renderer.hpp:436-478) and the ray-stream / BVH machinery under
 * them. The reference has no FFI of its own (one header-only C++ class template used directly by the app,
 * Application.cpp:373-382); these entry points are what a binding for that class would need, and the C++
 * mirror in cpu-raytracing-experiments_b200/host/ (Renderer.hpp, Scene.hpp, Camera.hpp, BVH.hpp) forwards
 * the reference's own member functions to them. INTEGRATION.md shows the reference-side change.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns B2R_OK (0) or a
 * negative B2R_ERR_* code and never throws; input arrays are caller-owned and copied during the call;
 * one host thread per context (the reference is single-threaded at this boundary, Application.cpp:361-382);
 * all device work of a context runs on one CUDA stream (b2r_set_stream). There is NO CPU fallback: without a
 * CUDA device every call that needs one fails with B2R_ERR_CUDA.
 */
#ifndef B2R_H_
#define B2R_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2R_ABI_VERSION 1

/* ---- PODs, layout-identical to the reference so its vectors can be passed as-is ---------------------- */
typedef struct b2r_sphere {      /* Sphere, Primitives.hpp:7-17 (alignas(16) => 32 B) */
	float position[3];
	float radius_sq;
	int32_t material_ID;
	int32_t _pad[3];
} b2r_sphere;

typedef struct b2r_material {    /* Material, Primitives.hpp:18-27 (alignas(32) => 96 B); hot path reads albedo + emission */
	float albedo[3], F0[3], F80[3], emission[3], transmission[3];
	float roughness, IOR_minus_one;
	float _pad[7];
} b2r_material;

typedef struct b2r_bvh_node {    /* BoundingVolumeHierarchy<Sphere>::Node, BVH.hpp:18-27 (32 B) */
	float min_bound[3];
	uint32_t first_id;           /* inner: index of the adjacent child pair; leaf: first primitive */
	float max_bound[3];
	uint32_t prim_count;         /* 0 = inner node, 1 = leaf (leaf size is always 1, BVH.hpp:133) */
} b2r_bvh_node;

/* ---- configuration (RendererPolicy NTTP + compile-time #defines of the reference, made run-time) ---- */
enum {
	B2R_FLAG_FORCE_BRUTE = 1u << 0, /* USEBVH false semantics at any scene size: test every ray against every sphere (BVH.hpp:311-318) */
	B2R_FLAG_FORCE_BVH   = 1u << 1, /* always use the flattened-BVH traversal kernels (default: brute <= 32 spheres, BVH above) */
	B2R_FLAG_NO_MIS      = 1u << 2, /* this repo's "MIS off" (SURVEY Q23): no light sampling, radiance += throughput*emission */
	B2R_FLAG_COUNT_TESTS = 1u << 3, /* also count sphere / box tests (slower; for roofline accounting) */
	B2R_FLAG_NO_GRAPH    = 1u << 4, /* launch kernels one by one instead of replaying a CUDA graph (profiling) */
	B2R_FLAG_REFERENCE_TREE = 1u << 5, /* traverse the flattened REFERENCE tree (BVH.hpp:90-206 topology) instead of the tree built for traversal */
	B2R_FLAG_REFERENCE_EXACT = 1u << 6, /* both pipelines, chosen at b2r_create: reproduce the reference's slot-dependent choice of sphere
	                                     * formula (BVH.hpp:250-286: the last `active % 8` rays of each 16x16 tile's stream take the scalar tail;
	                                     * stream order = stable counting sort by material, DataStreams.hpp:236-253). Results are then bit-identical
	                                     * to the reference's own Renderer::Accumulate, at the price of one extra ranking kernel per bounce. */
	B2R_FLAG_GPU_TREE = 1u << 8,       /* b2r_upload_scene builds the traversal tree ON THE GPU (Hilbert keys, radix sort, implicit balanced 4-ary topology, refit passes):
	                                    * milliseconds instead of the host's SAH build, for edits that add or remove spheres; same results, ~2x the node visits
	                                    * of the SAH tree on C3's overlapping spheres. May be toggled with b2r_set_flags between uploads. */
	B2R_FLAG_GPU_SAH = 1u << 10,       /* with B2R_FLAG_GPU_TREE: the device builds the SWEEP tree instead — the spheres stay in curve order and every node is a run of that
	                                    * order, cut top-down where the surface-area heuristic along the curve is smallest (segmented scans + one atomic minimum per
	                                    * run and round), opened 2 -> 4 wide like the host's collapse: ~1.1x the node visits of the host's SAH tree, built in ~1.2 ms of device time at 100k spheres. A scene whose sweep
	                                    * tree would be deeper than the traversal stack allows gets the packed tree. Node memory is reserved for the bound (one node per
	                                    * sphere), so the sweep flags take scenes of up to 2^22 spheres. */
	B2R_FLAG_GPU_SAH3 = 1u << 11,      /* with B2R_FLAG_GPU_TREE (wins over B2R_FLAG_GPU_SAH): the three-axis sweep — the device keeps the spheres sorted by centre x, y and z, every
	                                    * cut is the cheapest over all three orders (a full-sweep SAH build), the other two orders are partitioned to match: the node visits
	                                    * of the host's SAH tree, built on the device. Same depth fall-back as B2R_FLAG_GPU_SAH. */
	B2R_FLAG_GGX = 1u << 9,            /* the reference's `#define BRDF 1` build (Renderer.hpp:70,207-213): Closure<GGX> (DataStreams.hpp:184-219) from the materials'
	                                    * F0 and roughness instead of the Lambertian closure; gloss_decay_table (never declared by the reference) is all zeros and
	                                    * Closure<GGX>::pdf returns 0 as it does there. Not combinable with B2R_FLAG_REFERENCE_EXACT. */
	B2R_FLAG_NO_SPECULATION = 1u << 7, /* b2r_accumulate(ctx, 1) traces exactly one sample (default: a caller that asks for one sample per frame gets
	                                    * batches of 2, 4, ... 16 samples traced ahead while nothing changes; results are identical either way) */
	B2R_FLAG_DIELECTRIC = 1u << 12,    /* renders the materials' transmission and IOR, which the reference carries but never reads: a material with
	                                    * max(transmission) > 0 is a smooth dielectric of eta = 1 + IOR_minus_one (its albedo, F0, F80 and roughness are
	                                    * ignored). Each hit reflects with the Fresnel reflectance or refracts (throughput *= transmission), makes no light
	                                    * sample, and the emitter it reaches next gets MIS weight 1 (DESIGN.md §2). Other materials keep their closure; combines
	                                    * with B2R_FLAG_GGX, not with B2R_FLAG_REFERENCE_EXACT. With the flag, b2r_upload_scene, b2r_refit_scene and
	                                    * b2r_set_flags refuse (B2R_ERR_ARG) a non-finite transmission, and a dielectric with a transmission outside [0, 1]
	                                    * or an eta that is not finite or is < 1. A checkpoint does not load across the flag (b2r_load_checkpoint: B2R_ERR_STATE). */
	B2R_FLAG_SKY_LIGHT = 1u << 13,     /* samples the HDRI sky as a light (next-event estimation), combined with the BSDF-sampled misses by the power
	                                    * heuristic, in both pipelines (DESIGN.md §2). The sky is cut into the miss shader's cells, max(w-1,1) x max(h-1,1),
	                                    * drawn with probability ~ solid angle * (luminance of texel * ambient + its mean / 64) and uniformly in solid angle
	                                    * inside a cell; a light sample goes to the sky with probability 1 without sphere lights, 1/2 with them (a sphere
	                                    * light then has selection pdf 1 / (2 n_lights)). Lambertian surfaces only; a sample below the surface's horizon
	                                    * is dropped. The miss shader's contribution is per channel (quirk Q14 does not apply), and the path record then
	                                    * carries the local-cosine pdf of its direction (quirk Q10 does not apply). Quirk Q11 (a path that still hits at the
	                                    * last bounce loses its radiance) then also drops the sky's light samples of its earlier bounces, which without the
	                                    * flag never happens to sky light (it arrives only at a miss): at a finite max_bounces the flag-on image is lower in
	                                    * expectation by the energy those paths had gathered from the sky (DESIGN.md §2). Without a sky (ambient 0, or a texture
	                                    * that is zero everywhere) frames equal those without the flag. The sky's tables are built on the device at
	                                    * b2r_upload_scene, or when b2r_set_flags turns the flag on (b2r_read_sky_tables reads them). Combines with a lens
	                                    * and B2R_FLAG_DIELECTRIC; B2R_ERR_ARG with B2R_FLAG_REFERENCE_EXACT, B2R_FLAG_NO_MIS or B2R_FLAG_GGX, at b2r_create
	                                    * and b2r_set_flags. With the flag, b2r_upload_scene and b2r_set_flags refuse (B2R_ERR_ARG) a sky texel that is not
	                                    * finite, or negative, in a channel whose ambient is > 0. A checkpoint does not load across the flag. */
	B2R_FLAG_LIGHT_TREE = 1u << 14,    /* next-event estimation picks its sphere light by importance from a light tree instead of uniformly, in both
	                                    * pipelines (DESIGN.md §2). The tree is a binary tree over the light list, built on the host (median splits of the
	                                    * light centres, one light per leaf); a node keeps the box of its light spheres and its energy E = sum of
	                                    * mean(emission) * r^2. The sample's draw descends it by the importance E / max(|P - c|^2, R^2) of each child at the
	                                    * surface point; the light's selection pdf is (1 - p_sky) times the product of the branch probabilities, and an
	                                    * emissive hit recomputes that pdf at the point its light sample was taken from. The self test compares the picked
	                                    * light's BVH-order sphere with the hit sphere (quirk Q9 does not apply), the path record carries the local-cosine pdf
	                                    * of its direction whenever there are sphere lights (quirk Q10 does not apply), and an emitter that is not in the
	                                    * light list has selection pdf 0. Without sphere lights frames equal those without the flag. The tree is rebuilt at
	                                    * b2r_upload_scene and b2r_refit_scene, or when b2r_set_flags turns the flag on (b2r_read_light_tree reads it).
	                                    * Combines with B2R_FLAG_GGX, B2R_FLAG_DIELECTRIC, B2R_FLAG_SKY_LIGHT and a lens; B2R_ERR_ARG with
	                                    * B2R_FLAG_REFERENCE_EXACT or B2R_FLAG_NO_MIS, at b2r_create and b2r_set_flags. With the flag, b2r_upload_scene,
	                                    * b2r_refit_scene and b2r_set_flags refuse (B2R_ERR_ARG) a light list with a light index twice, or two lights that are
	                                    * equal spheres (position, radius^2, material), or a light whose emission is not finite or is negative. A checkpoint
	                                    * does not load across the flag. */
};

typedef struct b2r_config {
	uint32_t width, height;      /* multiples of 16 (Renderer::RequiredTiling(), Renderer.hpp:36) */
	uint32_t max_bounces;        /* RendererPolicy::max_bounces, Renderer.hpp:24 (reference: 16) */
	uint32_t buckets;            /* AccumulationBuckets, Renderer.hpp:41 (reference: 5); 1..64 */
	uint32_t flags;              /* B2R_FLAG_* */
	int32_t  device;             /* CUDA ordinal */
	uint32_t bucket_first;       /* multi-GPU: this context renders the samples whose bucket b = acc % buckets */
	uint32_t bucket_stride;      /*            satisfies b % bucket_stride == bucket_first (0/1 => all)   */
	uint32_t samples_in_flight;  /* samples the queue memory holds (<= 64); 0 = auto (~128M paths, 4..64). A wavefront batch traces up to this many together —
	                              * half of it on the BVH pipeline when the number is even: consecutive batches then alternate between the two halves ("sides")
	                              * and overlap on the device; inside a batch the samples may be traced as two lanes on two streams. Results never depend on it. */
} b2r_config;

enum {
	B2R_OK = 0,
	B2R_ERR_ARG = -1,            /* null pointer, size not a multiple of 16, bad bucket count, ... */
	B2R_ERR_CUDA = -2,           /* CUDA runtime error or no device (see b2r_last_error) */
	B2R_ERR_STATE = -3,          /* call order: e.g. accumulate before upload_scene */
	B2R_ERR_NO_LIGHTS = -4,      /* reserved: a scene without emissive spheres is accepted and simply gets no light sampling (SURVEY Q15) */
	B2R_ERR_BVH = -5,            /* malformed node array or traversal stack bound exceeded */
	B2R_ERR_NOT_READY = 1,       /* b2r_resolve: accumulations % buckets != 0 — Render() is a no-op then (Renderer.hpp:437) */
};

typedef struct b2r_ctx b2r_ctx;

/* ---- host-side scene preparation (replaces BVH.hpp:90-206 and Scene.hpp:12-16; runs on the CPU like the reference) */

/* BoundingVolumeHierarchy<Sphere>(span<const Sphere>) — BVH.hpp:90-206. nodes_out holds 2n-1 nodes (1 if n==0),
 * prims_out the spheres in leaf order (BVH.hpp:201-205), prim_ids_out[i] = geometry index of prims_out[i] (may be NULL). */
int b2r_bvh_build(const b2r_sphere* geometry, uint32_t n, b2r_bvh_node* nodes_out, b2r_sphere* prims_out,
                  uint32_t* prim_ids_out, uint32_t* n_nodes_out);
/* The same constructor with its second argument, SplitHeuristic{log_cluster_size, cost_ratio} (BVH.hpp:70-83, :90; the app always passes
 * the defaults {0, 1.0f}, which is what b2r_bvh_build uses): leaf cost = half_area * ceil(size / 2^log_cluster_size), the cost of not
 * splitting = half_area * (that count - cost_ratio). log_cluster_size <= 31. */
int b2r_bvh_build_ex(const b2r_sphere* geometry, uint32_t n, uint32_t log_cluster_size, float cost_ratio, b2r_bvh_node* nodes_out,
                     b2r_sphere* prims_out, uint32_t* prim_ids_out, uint32_t* n_nodes_out);
/* LightingAcceleration(geometry, material) — Scene.hpp:12-16. Returns the count via n_out; out may be NULL to size. */
int b2r_find_lights(const b2r_sphere* geometry, uint32_t n, const b2r_material* materials, uint32_t n_mat,
                    int32_t* out, uint32_t* n_out);
/* View(eye, forward) + Projection::Resize/UpdateLens — Camera.hpp:21-32,47-50. out11 = pos[3], orient wxyz[4],
 * half_width, half_height, z, exposure: the exact arguments of b2r_set_camera. */
int b2r_camera_lookat(const float eye[3], const float dir[3], uint32_t width, uint32_t height, float focal_length_mm,
                      float exposure, float out11[11]);

/* Camera::generate_ray (Camera.hpp:80-88) for ONE pixel, on the host: view.pos and normalize(view.orient * {x + samples[0] - half_width,
 * y + samples[1] - half_height, z}) with glm's scalar arithmetic — the call the app's focus picking makes (Application.cpp:288) before it
 * hands the ray to BoundingVolumeHierarchy::Traverse (b2r_trace_closest). The renderer's own camera rays are generated on the GPU by the
 * same routine (b2r_generate_rays); this entry is for host code that needs a single ray. */
int b2r_camera_ray(const float pos[3], const float orient_wxyz[4], float half_width, float half_height, float z,
                   int32_t x, int32_t y, const float samples[2], float origin_out[3], float dir_out[3]);

/* ---- renderer life cycle (Renderer<Policy>, Renderer.hpp:28-68) -------------------------------------- */
int  b2r_create(b2r_ctx** out, const b2r_config* cfg);             /* Renderer(const Scene&) + Resize, :51-63 */
void b2r_destroy(b2r_ctx* ctx);
int  b2r_resize(b2r_ctx* ctx, uint32_t width, uint32_t height);     /* Renderer::Resize, :53-63 (resets the accumulator) */
int  b2r_reset(b2r_ctx* ctx);                                       /* Renderer::ResetAccumulator, :64-67 */
int  b2r_set_stream(b2r_ctx* ctx, void* cuda_stream);               /* run on a caller-owned cudaStream_t (NULL = own stream) */
int  b2r_sync(b2r_ctx* ctx);

/* Scene (Scene.hpp:19-26) as the renderer reads it: spheres in BVH leaf order + nodes (acceleration_structure),
 * materials, the light list (indices into geometry) and geometry in original order (read by NEE, Renderer.hpp:261-262),
 * sky (Primitives.hpp:29-47; hdri_rgba may be NULL when ambient is 0). The node array is validated; the GPU traverses a 128-byte
 * 4-wide layout whose leaves are exactly prims_bvh_order (hit indices are BVH-order indices). By default its topology is rebuilt
 * for traversal speed (results do not depend on it: closest hit == brute force); B2R_FLAG_REFERENCE_TREE flattens `nodes` itself.
 * The derived layout is cached per context and reused while the spheres are unchanged. */
int  b2r_upload_scene(b2r_ctx* ctx, const b2r_sphere* prims_bvh_order, const b2r_bvh_node* nodes, uint32_t n_prims,
                      uint32_t n_nodes, const b2r_material* materials, uint32_t n_mat, const int32_t* light_geom_idx,
                      uint32_t n_lights, const b2r_sphere* geometry, uint32_t n_geom, const float ambient[3],
                      const float* hdri_rgba, int32_t hdri_w, int32_t hdri_h);
/* Scene edit without rebuilding the traversal tree. The reference rebuilds its BVH on every geometry drag (Application.cpp:508-509, then
 * ResetAccumulator :510). Here the spheres keep their count and move / change radius or material; prims_bvh_order is either the order
 * of the last upload or a NEW one (the reference's constructor re-sorts its prims on every rebuild, BVH.hpp:201-205, and hit indices,
 * Q6 ties and the Q9 self-test are defined on that order) — it only has to be a permutation of `geometry`, which is how the library
 * finds out which sphere went where (matched by value; the reference's BVH keeps no index map). The packed spheres and the light table
 * are uploaded again; the traversal tree keeps its TOPOLOGY, its leaves are re-linked to the new order and its boxes are recomputed ON
 * THE GPU, bottom-up, one launch per tree level (k_refit_level) — asynchronous on the context's stream, no host tree build, the captured
 * CUDA graph stays valid. Results are those of a fresh b2r_upload_scene of the same arrays (closest hit == brute force over
 * prims_bvh_order); only the tree's speed depends on how far the spheres moved from where it was built. quality_out (may be NULL;
 * asking costs one more launch and a stream synchronisation) = sum of the inner boxes' surface areas now / when the tree was built:
 * rebuild with b2r_upload_scene once it grows past ~1.5. B2R_ERR_STATE before the first upload; B2R_ERR_ARG when the count changed or
 * prims_bvh_order is not a permutation of geometry. The caller resets the accumulator (b2r_reset) as the reference does. */
int  b2r_refit_scene(b2r_ctx* ctx, const b2r_sphere* prims_bvh_order, uint32_t n_prims, const b2r_material* materials, uint32_t n_mat,
                     const int32_t* light_geom_idx, uint32_t n_lights, const b2r_sphere* geometry, uint32_t n_geom, float* quality_out);
/* Camera (Camera.hpp:61-88): view.pos, view.orient (w,x,y,z), projection.half_width/half_height/z, exp */
int  b2r_set_camera(b2r_ctx* ctx, const float pos[3], const float orient_wxyz[4], float half_width, float half_height,
                    float z, float exposure);
/* Thin-lens depth of field (opt-in; the reference computes Projection::aperture_radius but renders a pinhole, Camera.hpp:80-88).
 * lens_radius R and focus_distance F are in SCENE UNITS: the library does not guess a millimetre-to-scene scale, the caller converts
 * (aperture_radius = focal_length / (2 f_number) is in mm). F is measured along the camera's forward axis: the plane camera-space
 * z = -F is in focus. Camera ray = from pos + orient * L, L a point of the lens disk of radius R, through the point where the pinhole ray
 * of the same pixel sample meets that plane. R = 0 (the default) is the pinhole camera, bit for bit. Takes effect like b2r_set_camera
 * (batches already enqueued keep their lens). b2r_camera_ray stays the pinhole ray through the lens centre (focus picking).
 * B2R_ERR_ARG: R negative or not finite, F not finite or <= 0. B2R_ERR_STATE: a B2R_FLAG_REFERENCE_EXACT context. */
int  b2r_set_lens(b2r_ctx* ctx, float lens_radius, float focus_distance);

/* ---- the hot path ---------------------------------------------------------------------------------- */
/* Renderer::Accumulate() n_samples times (Renderer.hpp:73-434): accumulations += n_samples; each new sample index
 * acc lands in bucket acc % buckets (this context renders only the buckets it owns). Asynchronous on the stream. */
int  b2r_accumulate(b2r_ctx* ctx, uint32_t n_samples);
/* Renderer::Render() (Renderer.hpp:436-478): median-of-K bucket sums * exposure/(accumulations/K), ACES tonemap
 * (tonemap=0: linear), RGBA32F, row 0 = y 0. rgba_out_host: width*height*4 floats (NULL: leave it on the device).
 * Returns B2R_ERR_NOT_READY and writes nothing unless accumulations % buckets == 0. Synchronises. */
int  b2r_resolve(b2r_ctx* ctx, float* rgba_out_host, int tonemap);
/* Render() without the stall: the resolve kernel is enqueued on the context's stream and the frame is copied to rgba_out_host on a
 * second stream, so the next b2r_accumulate calls overlap the copy (progressive rendering: frame N leaves while the samples of
 * frame N+1 are traced). rgba_out_host must be page-locked for the overlap and must stay valid until b2r_frame_wait() returns;
 * a following resolve waits (on the device) for the pending copy before it overwrites the device framebuffer.
 * Returns B2R_ERR_NOT_READY like b2r_resolve. The reference's Render() is synchronous (Renderer.hpp:436-478); this is the same
 * computation with the hand-over made explicit. */
int  b2r_resolve_async(b2r_ctx* ctx, float* rgba_out_host, int tonemap);
int  b2r_frame_wait(b2r_ctx* ctx);   /* blocks until the frame of the last b2r_resolve_async has landed in host memory */
/* Render() into the device framebuffer (b2r_device_framebuffer) without waiting for it: only enqueues the resolve kernel, so frames enqueued
 * back to back are pipelined on the device — the library traces consecutive batches on alternating halves of its queue memory ("sides"), and
 * the thin last bounces of frame N, its fold and its resolve run under the first bounces of frame N+1. b2r_sync (or any synchronising call)
 * before the frame is read. Same return values as b2r_resolve. */
int  b2r_resolve_device(b2r_ctx* ctx, int tonemap);
/* Same, reading the K bucket sums from another device array of the same layout (e.g. the NCCL-combined buckets of a
 * multi-GPU frame) instead of this context's own accumulator. dev_buckets == NULL means the context's own. */
int  b2r_resolve_from(b2r_ctx* ctx, const void* dev_buckets, float* rgba_out_host, int tonemap);

/* Page-lock a caller-owned frame buffer (the reference's `framebuffer` vector, Renderer.hpp:40) so that b2r_resolve's copy into it runs at
 * DMA speed instead of through the driver's staging path (33 MB at 1080p: ~1 ms instead of ~4 ms). The C++ faces do this after Resize. */
int  b2r_host_register(void* ptr, size_t bytes);
int  b2r_host_unregister(void* ptr);

/* ---- taps: parity, metrics, resume, multi-GPU plumbing --------------------------------------------- */
int  b2r_get_accumulations(b2r_ctx* ctx, uint32_t* out);
int  b2r_set_accumulations(b2r_ctx* ctx, uint32_t acc);            /* resume / jump to a sample index (RNG is stateless, Q2-Q3) */
int  b2r_read_buckets(b2r_ctx* ctx, float* out_host);               /* [buckets][3][width*height], pixels in tile order t = tile*256+ID */
int  b2r_write_buckets(b2r_ctx* ctx, const float* in_host);         /* checkpoint restore */
/* Checkpoint / resume of a progressive render as ONE file: a 64-byte header (magic, frame size, bucket count, bounce limit, accumulations,
 * the flags that change the image, payload size and hash) followed by the bucket sums exactly as b2r_read_buckets returns them. Loading
 * checks all of it (B2R_ERR_ARG: not a checkpoint / truncated / corrupt; B2R_ERR_STATE: written for another configuration) and then
 * restores the buckets and the sample counter, so that further b2r_accumulate calls continue the SAME image bit for bit (the RNG is a pure
 * function of sample index, pixel and bounce, Q2-Q3). The reference has no such file: its only dump is the tonemapped frame (Image.cpp:71-74). */
int  b2r_save_checkpoint(b2r_ctx* ctx, const char* path);
int  b2r_load_checkpoint(b2r_ctx* ctx, const char* path);
int  b2r_device_buckets(b2r_ctx* ctx, void** dev_ptr, size_t* bytes); /* device address of the same array (NCCL / P2P combine) */
int  b2r_device_framebuffer(b2r_ctx* ctx, void** dev_ptr, size_t* bytes);
/* Multi-GPU resolve over peer memory (NVLink P2P), the fused alternative to combine-then-resolve: every process exports its
 * bucket array as a 64-byte CUDA IPC handle, exchanges the handles (any transport), opens its peers' arrays, and the resolve
 * kernel reads bucket k straight from its owner's HBM (owner = k % n_peers, b2r_config.bucket_*), so no bucket is copied or
 * reduced first. Callers must order the resolve after every peer's b2r_sync (one barrier). peer_handles: n_peers x 64 bytes in
 * rank order (the entry of `my_rank` is ignored). b2r_ipc_close drops the mappings. */
int  b2r_ipc_export_buckets(b2r_ctx* ctx, unsigned char handle_out[64]);
int  b2r_ipc_open_peers(b2r_ctx* ctx, const unsigned char* peer_handles, uint32_t n_peers, uint32_t my_rank);
int  b2r_ipc_close(b2r_ctx* ctx);
int  b2r_resolve_peers(b2r_ctx* ctx, float* rgba_out_host, int tonemap);
/* Team mode — the multi-GPU frame without host barriers. Every rank exports three handles (its bucket array, its framebuffer, a small
 * block of hand-shake flags), the ranks exchange them once (any transport) and open each other's; after that a frame needs no host
 * synchronisation between ranks at all. b2r_team_resolve, called by EVERY rank once its samples are enqueued: rank g waits on the device
 * until every rank's buckets of this frame are final, resolves the g-th slab of 16x16 tiles — median of the K bucket sums read straight
 * from their owners' HBM over NVLink (bucket k lives on rank k % n_ranks), exposure scale, ACES — and stores it into RANK 0's framebuffer
 * over NVLink; rank 0 then copies the frame to rgba_out_host (async != 0: on its copy stream, page-locked buffer, b2r_frame_wait to join;
 * NULL: the frame stays on the device). The hand-shakes are release/acquire flags in peer-mapped memory written and polled by tiny
 * kernels in stream order (a wait gives up after ~4 s and raises b2r_team_error instead of hanging the GPU); b2r_reset / b2r_accumulate
 * of the next frame wait the same way until the peers have finished reading this rank's buckets. The resolved frame is bit-identical to a
 * single-GPU render of the same samples. The resized framebuffer / bucket array must not be exported: b2r_resize fails while a team is open. */
int  b2r_team_export(b2r_ctx* ctx, unsigned char handles_out[192]);
int  b2r_team_open(b2r_ctx* ctx, const unsigned char* all_handles /* n_ranks x 192 bytes, rank order */, uint32_t n_ranks, uint32_t my_rank);
int  b2r_team_resolve(b2r_ctx* ctx, float* rgba_out_host, int tonemap, int async);
int  b2r_team_error(b2r_ctx* ctx, uint32_t* error_out);   /* 0 = no hand-shake has timed out (synchronises the stream) */
int  b2r_team_close(b2r_ctx* ctx);
/* counters since the last reset: [0] extension rays, [1] shadow rays, [2] shaded hits, [3] terminated paths,
 * [4] dropped at max_bounces (Q11), [5] sphere tests, [6] box tests (5,6 only with B2R_FLAG_COUNT_TESTS), [7] kernel launches,
 * [8] radiance contributions written (light samples, emissive hits, sky), [9] reserved */
int  b2r_read_counters(b2r_ctx* ctx, uint64_t out[10]);
int  b2r_reset_counters(b2r_ctx* ctx);
/* rays of the LAST wavefront batch per bounce: paths_out[b] = extension rays entering bounce b, shadow_out[b] = shadow rays queued at bounce b
 * (n entries each; what the per-launch roofline rows divide by). Synchronises. */
int  b2r_read_bounce_counts(b2r_ctx* ctx, uint32_t* paths_out, uint32_t* shadow_out, uint32_t n);
/* per-kernel device time (ms) and launch counts accumulated while B2R_FLAG_NO_GRAPH profiling is on:
 * index 0 generate, 1 bounce_brute, 2 intersect_closest, 3 shade, 4 intersect_shadow, 5 accumulate, 6 resolve */
int  b2r_read_kernel_times(b2r_ctx* ctx, double ms_out[8], uint64_t launches_out[8], int reset);
int  b2r_set_flags(b2r_ctx* ctx, uint32_t flags);

/* Camera::generate_ray for every pixel of sample index acc (Renderer.hpp:113-127): out_host[t*6 + {o.xyz, d.xyz}] */
int  b2r_generate_rays(b2r_ctx* ctx, uint32_t acc, float* out_host);
/* BoundingVolumeHierarchy::Traverse / Traverse_shadow on caller rays (public surface, Application.cpp:282-298):
 * rays_host[n*6] = origin, dir. closest: tfar_out[n] (FLT_MAX on miss), prim_out[n] (BVH-order index or -1). */
int  b2r_trace_closest(b2r_ctx* ctx, const float* rays_host, uint32_t n, float* tfar_out, int32_t* prim_out);
int  b2r_trace_shadow(b2r_ctx* ctx, const float* rays_host, const float* tfar_host, uint32_t n, uint8_t* occluded_out);
/* The traversal kernels a frame uses, on caller input (tests): the instantiation and grid the context's flags and scene select for a
 * frame, run on queue buffers of the call's own, so nothing of the renderer's state (queues, samples traced ahead, counters) is touched.
 * B2R_ERR_STATE before an upload or on a brute-force context; B2R_ERR_ARG for a null pointer the kernel needs or an unknown kernel.
 *  B2R_TAP_CLOSEST  k_intersect_closest: rays[n*6] -> tfar_out[n], prim_out[n] (as b2r_trace_closest). tail: NULL or n bytes; with
 *                   B2R_FLAG_REFERENCE_EXACT, nonzero = this ray takes the scalar-tail sphere formula (BVH.hpp:270-286).
 *                   origin_prim: NULL (every walk starts at the root) or n entries, as for B2R_TAP_SHADOW: ray i's walk starts at the
 *                   wide node holding sphere origin_prim[i], or at the root for -1, and climbs (B2R_ERR_ARG for an index >= the sphere count).
 *  B2R_TAP_SHADOW   k_intersect_shadow: rays, tfar[n] -> occluded_out[n]; ray i's walk starts at the wide node holding sphere
 *                   origin_prim[i] (BVH order), or at the root for -1, and climbs (B2R_ERR_ARG for an index >= the sphere count).
 *  B2R_TAP_PACKET   k_intersect_packet on the camera rays of sample index acc (rays unused): n == width*height (else B2R_ERR_ARG),
 *                   tfar_out / prim_out in tile order, entry t being ray t of b2r_generate_rays(acc). */
enum { B2R_TAP_CLOSEST = 0, B2R_TAP_SHADOW = 1, B2R_TAP_PACKET = 2 };
int  b2r_trace_kernel(b2r_ctx* ctx, int kernel, const float* rays, const float* tfar, const int32_t* origin_prim, const uint8_t* tail,
                      uint32_t n, uint32_t acc, float* tfar_out, int32_t* prim_out, uint8_t* occluded_out);
/* the flattened 128-byte node array (for the layout round-trip test): out may be NULL to size */
int  b2r_read_wide_nodes(b2r_ctx* ctx, void* out_host, uint32_t* n_wide_nodes, uint32_t* max_stack);
/* the link tables k_link_tables derives from the device tree: parent_out[n_wide_nodes] (the node that links to node i, 0 for the root)
 * and leaf_node_out[n_prims] (the node whose leaf slot holds sphere i, BVH order). Synchronises. */
int  b2r_read_link_tables(b2r_ctx* ctx, uint32_t* parent_out, uint32_t* leaf_node_out);
/* B2R_FLAG_SKY_LIGHT: the sky's tables as the device built them. *cols_out = W' = max(w-1,1), *rows_out = H' = max(h-1,1); marginal_out[H'+1]
 * (CDF over the rows), conditional_out[H'][W'+1] (CDF over the cells of each row), pdf_out[h][w] (solid-angle pdf of the cell each texel shows,
 * without the sky's selection probability). A null table pointer skips that table. B2R_ERR_STATE when no tables are built. Synchronises. */
int  b2r_read_sky_tables(b2r_ctx* ctx, float* marginal_out, float* conditional_out, float* pdf_out, uint32_t* cols_out, uint32_t* rows_out);
/* B2R_FLAG_LIGHT_TREE: the light tree as the device holds it. *n_nodes_out = its node count N (2 n_lights - 1); nodes_out[N][8] = per node
 * {c.x, c.y, c.z, R^2, E, link, 0, 0}: the box of its light spheres as centre and squared half-diagonal, its energy, and `link` (an int32 stored
 * in the float's bits): >= 0, the children are nodes link and link + 1; < 0, a leaf holding light ~link. Node 0 is the root.
 * light_prim_out[n_lights] = the BVH-order sphere of each light (the lowest index equal to it by value; -1: none). A null table pointer skips
 * that table. B2R_ERR_STATE when no tree is built (the flag is off, or the scene has no sphere lights). Synchronises. */
int  b2r_read_light_tree(b2r_ctx* ctx, float* nodes_out, int32_t* light_prim_out, uint32_t* n_nodes_out);
/* the box ray origins are assumed to lie in ({lo.xyz, hi.xyz}: sphere bounds, camera, origins passed to b2r_trace_*): the leaf slots of the
 * traversal tree are sized for it, so a host twin of the tree needs the same box (tests) */
int  b2r_get_origin_box(b2r_ctx* ctx, float lo_hi_out[6]);

/* Image::Store (Image.cpp:71-74 -> stbi_write_hdr with vertical flip, called on F5, Application.cpp:254-257): writes the
 * RGBA32F framebuffer as a Radiance .hdr (32-bit_rle_rgbe, rows written top-down = framebuffer rows in reverse, alpha dropped). */
int  b2r_write_hdr(const char* path, const float* rgba, uint32_t width, uint32_t height);

/* The sky texture as the reference loads it: stbi_loadf(path, &w, &h, &channels, 4) (Application.cpp:225-231) — a Radiance .hdr
 * (32-bit_rle_rgbe, "-Y h +X w") decoded to RGBA32F rows in file order, channel = mantissa * 2^(e-136), alpha 1; exactly the array
 * b2r_upload_scene takes as hdri_rgba. rgba_out may be NULL to query the size first. B2R_ERR_ARG for a file stb_image would reject
 * (not Radiance, other FORMAT or orientation, corrupt run lengths) and for a truncated one. */
int  b2r_read_hdr(const char* path, float* rgba_out, int32_t* width_out, int32_t* height_out);

const char* b2r_last_error(void);   /* text of the last failure on this thread */
int  b2r_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B2R_H_ */
