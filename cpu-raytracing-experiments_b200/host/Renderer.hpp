// Renderer.hpp — drop-in for the reference's Renderer<Policy> (Renderer.hpp:28-479): same public members and call sequence
// (Application.cpp:373-382: Resize -> Accumulate -> Render -> read framebuffer), forwarding to the C ABI of libb2r.so.
//
// Differences a caller can see, all forced by the device boundary:
//   * `framebuffer` is filled by Render() from the GPU (RGBA32F, tonemapped, row 0 = y 0) — there is no Vulkan Image; GetFrame()
//     returns the framebuffer vector instead of unique_ptr<Image>;
//   * the reference reads `const Scene&` live; here the scene is snapshotted at construction and after SceneChanged() (the app
//     already calls ResetAccumulator() at exactly those points, Application.cpp:508-510);
//   * Policy is a run-time struct (same field names and defaults), AccumulationBuckets is Policy.buckets (reference: 5);
//   * failures throw std::runtime_error with libb2r's message (the reference has no error path at all).
#pragma once
#include <stdexcept>
#include <string>
#include <vector>
#include "Camera.hpp"
#include "Primitives.hpp"
#include "BVH.hpp"

// ---- the data model the renderer borrows (Scene.hpp:9-26): the light list is built by libb2r, the aggregate keeps the
// reference's member names so that Application.cpp:33-101,233-234 compiles unchanged
struct LightingAcceleration {  // Scene.hpp:9-17: indices (into scene.geometry) of the emissive spheres
	std::vector<int32_t> prims;
	LightingAcceleration() {}
	LightingAcceleration(const std::vector<Sphere>& src_prims, const std::vector<Material>& material) {
		uint32_t n = 0;
		prims.resize(src_prims.size());
		b2r_find_lights(reinterpret_cast<const b2r_sphere*>(src_prims.data()), static_cast<uint32_t>(src_prims.size()),
		                reinterpret_cast<const b2r_material*>(material.data()), static_cast<uint32_t>(material.size()), prims.data(), &n);
		prims.resize(n);
	}
};

struct Scene {  // Scene.hpp:19-26
	std::vector<Sphere> geometry;
	std::vector<Material> material;
	LightingAcceleration lighting_acceleration;
	Camera camera;
	Sky sky;
	BoundingVolumeHierarchy<Sphere> acceleration_structure;
};

struct RendererPolicy {  // Renderer.hpp:19-26
	size_t log_tile = 4;
	size_t samples_per_pixel = 1;
	size_t max_materialID = 64;
	size_t max_bounces = 16;
	float max_radiance = 1e2f;   // unused by the reference as well (Q5)
	size_t buckets = 5;          // AccumulationBuckets, Renderer.hpp:41
	uint32_t flags = 0;          // B2R_FLAG_*
	int device = 0;
};

struct Renderer {
	RendererPolicy Policy;
	static constexpr size_t TileRoot = 16, TileSize = 256, StreamSize = 256;
	static constexpr size_t RequiredTiling() { return TileRoot; }  // Renderer.hpp:36

	const Scene& scene;
	std::vector<b2r_host::vec4> framebuffer;
	uint32_t width = 0, height = 0;
	uint32_t accumulations = 0;
	uint32_t h_tiles = 0, v_tiles = 0;

	explicit Renderer(const Scene& scene, RendererPolicy policy = {}) : Policy(policy), scene(scene) {}
	~Renderer() { if (!framebuffer.empty()) b2r_host_unregister(framebuffer.data()); if (ctx) b2r_destroy(ctx); }
	Renderer(const Renderer&) = delete;
	Renderer& operator=(const Renderer&) = delete;

	void Resize(uint32_t new_width, uint32_t new_height) {  // Renderer.hpp:53-63
		height = new_height; width = new_width;
		if (!framebuffer.empty()) b2r_host_unregister(framebuffer.data());
		framebuffer.resize(static_cast<size_t>(width) * height);
		b2r_host_register(framebuffer.data(), framebuffer.size() * sizeof(framebuffer[0]));  // Render() copies into it at DMA speed (best effort)
		h_tiles = width / TileRoot; v_tiles = height / TileRoot;
		if (!ctx) {
			b2r_config cfg{}; cfg.width = width; cfg.height = height; cfg.max_bounces = static_cast<uint32_t>(Policy.max_bounces);
			cfg.buckets = static_cast<uint32_t>(Policy.buckets); cfg.flags = Policy.flags; cfg.device = Policy.device;
			check(b2r_create(&ctx, &cfg));
			SceneChanged();
		} else check(b2r_resize(ctx, width, height));
		accumulations = 0;
		CameraChanged();
	}
	void ResetAccumulator() { accumulations = 0; check(b2r_reset(ctx)); CameraChanged(); }  // Renderer.hpp:64-67 (callers reset after moving the camera)
	auto& GetFrame() { return framebuffer; }  // Renderer.hpp:68

	// re-snapshot geometry / materials / BVH / lights after an edit (Application.cpp:508-510 rebuilds them, then resets)
	void SceneChanged() {
		const auto& as = scene.acceleration_structure;
		const float amb[3] = {scene.sky.ambient_color.x, scene.sky.ambient_color.y, scene.sky.ambient_color.z};
		check(b2r_upload_scene(ctx, reinterpret_cast<const b2r_sphere*>(as.prims.data()), as.nodes.data(), static_cast<uint32_t>(as.prims.size()),
		                       static_cast<uint32_t>(as.nodes.size()), reinterpret_cast<const b2r_material*>(scene.material.data()),
		                       static_cast<uint32_t>(scene.material.size()), scene.lighting_acceleration.prims.data(),
		                       static_cast<uint32_t>(scene.lighting_acceleration.prims.size()), reinterpret_cast<const b2r_sphere*>(scene.geometry.data()),
		                       static_cast<uint32_t>(scene.geometry.size()), amb, scene.sky.hdri_data, scene.sky.hdri_width, scene.sky.hdri_height));
	}
	// geometry moved and the app has rebuilt acceleration_structure / lighting_acceleration (Application.cpp:508-509): the GPU keeps its
	// traversal tree's topology, re-links the leaves to the rebuilt order and refits the boxes (b2r_refit_scene) instead of rebuilding;
	// full SceneChanged() when the sphere count changed or the kept topology degraded past `rebuild_above`. Returns the quality ratio.
	float SceneMoved(float rebuild_above = 1.5f) {
		const auto& as = scene.acceleration_structure;
		float quality = 1.0f;
		const int rc = b2r_refit_scene(ctx, reinterpret_cast<const b2r_sphere*>(as.prims.data()), static_cast<uint32_t>(as.prims.size()),
		                               reinterpret_cast<const b2r_material*>(scene.material.data()), static_cast<uint32_t>(scene.material.size()),
		                               scene.lighting_acceleration.prims.data(), static_cast<uint32_t>(scene.lighting_acceleration.prims.size()),
		                               reinterpret_cast<const b2r_sphere*>(scene.geometry.data()), static_cast<uint32_t>(scene.geometry.size()), &quality);
		if (rc == B2R_ERR_ARG || rc == B2R_ERR_STATE || (rc == B2R_OK && quality > rebuild_above)) { SceneChanged(); return 1.0f; }
		check(rc);
		return quality;
	}
	void CameraChanged() {
		const Camera& c = scene.camera;
		const float pos[3] = {c.view.pos.x, c.view.pos.y, c.view.pos.z}, q[4] = {c.view.orient.w, c.view.orient.x, c.view.orient.y, c.view.orient.z};
		check(b2r_set_camera(ctx, pos, q, c.projection.half_width, c.projection.half_height, c.projection.z, c.exp));
	}
	// Thin-lens depth of field (b2r_set_lens), in scene units: the app's focus pick gives the distance; Projection::aperture_radius is in mm and
	// the caller scales it to scene units. lens_radius 0 = the pinhole camera.
	void SetLens(float lens_radius, float focus_distance) { check(b2r_set_lens(ctx, lens_radius, focus_distance)); }

	void Accumulate() { ++accumulations; check(b2r_accumulate(ctx, 1)); }             // Renderer.hpp:73-434
	void Accumulate(uint32_t n) { accumulations += n; check(b2r_accumulate(ctx, n)); } // n calls in one submission
	void Render() {                                                                    // Renderer.hpp:436-478
		const int rc = b2r_resolve(ctx, reinterpret_cast<float*>(framebuffer.data()), 1);
		if (rc < 0) check(rc);  // B2R_ERR_NOT_READY (accumulations % buckets != 0) is the reference's silent early return (:437)
	}
	// Render() into the DEVICE framebuffer without waiting (b2r_resolve_device): for a display path that reads device memory (b2r_device_framebuffer);
	// frames enqueued back to back are pipelined on the device. Sync() before the frame is read.
	void RenderDevice() { const int rc = b2r_resolve_device(ctx, 1); if (rc < 0) check(rc); }
	void Sync() { check(b2r_sync(ctx)); }
	// BoundingVolumeHierarchy::Traverse on caller rays (focus picking, Application.cpp:282-298): rays = n x {origin, dir}
	void Traverse(const float* rays, uint32_t n, float* tfar_out, int32_t* prim_out) { check(b2r_trace_closest(ctx, rays, n, tfar_out, prim_out)); }
	// BoundingVolumeHierarchy::Traverse_shadow (BVH.hpp:362): occluded_out[i] = 1 when anything lies within [0, tfar[i]) along ray i
	void Traverse_shadow(const float* rays, const float* tfar, uint32_t n, uint8_t* occluded_out) { check(b2r_trace_shadow(ctx, rays, tfar, n, occluded_out)); }
	b2r_ctx* handle() { return ctx; }

private:
	b2r_ctx* ctx = nullptr;
	static void check(int rc) { if (rc < 0) throw std::runtime_error(std::string("libb2r: ") + b2r_last_error()); }
};
