// b2r_shade.h — per-path shading and BVH traversal routines of the wavefront path tracer, host+device.
//
// The sm_100a kernels (b2r_device.cuh) call these from their persistent loops. They are also plain C++ so that
// tests/hostcheck can run the very same routines on the build box (which has no GPU) and compare them bit-for-bit
// with the oracle; nothing in libb2r.so executes them on the CPU (the one exception is bookkeeping, not rendering: slot_half_area()
// in the flattener's tree-cost sum).
#pragma once
#include <vector_types.h>
#include <vector_functions.h>
#include "b2r_math.h"
#include "b2r_host.h"

namespace b2r {

constexpr int kMaxSlots = 64;          // samples in flight per batch (pid keeps 6 slot bits)
constexpr uint32_t kPixMask = (1u << 26) - 1u;

B2R_HD int32_t as_int(float f) { return static_cast<int32_t>(bits(f)); }
B2R_HD float from_int(int32_t v) { return from_bits(static_cast<uint32_t>(v)); }
// read-only global data (BVH nodes): LDG through the read-only path
B2R_HD float4 ldg4(const float4* p) {
#if defined(__CUDA_ARCH__)
	return __ldg(p);
#else
	return *p;
#endif
}
B2R_HD uint32_t ldg_u32(const uint32_t* p) {
#if defined(__CUDA_ARCH__)
	return __ldg(p);
#else
	return *p;
#endif
}
// scene tables (spheres, materials, lights): generic loads, because the brute-force kernels point SceneDev at shared-memory copies
B2R_HD float4 ld4(const float4* p) { return *p; }

enum Stat { ST_EXT = 0, ST_SHADOW, ST_HITS, ST_TERM, ST_DROPPED, ST_SPHERE, ST_BOX, ST_EVENTS, ST_COUNT };

struct SceneDev {
	const float4* prims;        // [n_prims] {c.xyz, r^2}, BVH leaf order (acceleration_structure.prims)
	const int32_t* prim_mat;    // [n_prims] material_ID
	const float4* mat_albedo;   // [n_mat] {albedo.rgb, emissive ? 1 : 0}  (max(emission) > FLT_EPSILON, Renderer.hpp:201)
	const float4* mat_emission; // [n_mat] {emission.rgb, 0}
	const float4* mat_f0;       // [n_mat] {F0.rgb, roughness}: read by the GGX closure only (B2R_FLAG_GGX)
	const float4* light_sphere; // [n_lights] scene.geometry[light] {c.xyz, r^2}   (Renderer.hpp:261-262)
	const float4* light_emit;   // [n_lights] {emission.rgb of its material, as_float(light_primID)}
	const WideNode* wide;       // flattened BVH
	const uint32_t* parent;     // [n_wide] the wide node that links to node i (the root's entry is 0)      } written by k_link_tables from the device tree itself; the walks
	const uint32_t* leaf_node;  // [n_prims] the wide node that holds sphere i (BVH order) in a leaf slot       } of k_intersect_shadow and k_intersect_closest start there
	const float4* hdri;         // equirect RGBA32F or null
	uint32_t n_prims, n_mat, n_lights;
	uint32_t stack_tn_bits;     // traversal stack entry split (WideBvh::tn_bits)
	float light_sel_pdf;        // 1 / n_lights (Renderer.hpp:78)
	float ambient[3]; int32_t has_ambient;  // Renderer.hpp:79
	int32_t hdri_w, hdri_h; float hdri_fw, hdri_fh;
};
struct FrameDev {
	CameraParams cam;
	uint32_t width, height, h_tiles, npix;
	uint32_t max_bounces, buckets, flags;
	uint32_t h_tiles_magic, npix_magic;  // floor(2^32 / d) for div_by()
	uint32_t finish_below, finish_first;  // brute-force pipeline: once fewer than finish_below paths enter a bounce >= finish_first, k_brute_finish traces them to their end in one launch (0 = never)
};
// x / d for a launch-constant divisor without the ~20-instruction integer division: q = mulhi(x, floor(2^32/d)) is q or q-1.
B2R_HD uint32_t div_by(uint32_t x, uint32_t d, uint32_t magic) {
#if defined(__CUDA_ARCH__)
	uint32_t q = __umulhi(x, magic);
#else
	uint32_t q = static_cast<uint32_t>((static_cast<uint64_t>(x) * magic) >> 32);
#endif
	if (x - q * d >= d) q++;
	return q;
}
B2R_HD uint32_t magic_for(uint32_t d) { return d <= 1u ? 0xffffffffu : static_cast<uint32_t>((1ull << 32) / d); }
struct BatchDev {  // one wavefront batch: n_slots samples traced together
	uint32_t n_slots;
	uint32_t acc[kMaxSlots];  // sample index (the reference's `accumulations` value, Q1) of each slot
	CameraParams cam;         // the camera this batch is traced with: it travels with the batch descriptor (written by k_set_batch in front of every batch),
	                          // not with the kernels' parameter block, so a camera move neither re-captures the batch graph nor waits for the stream
	LensParams lens;          // likewise (read by the LENS instantiations only; a pinhole <-> lens switch changes the instantiation and re-captures)
	unsigned long long fold;  // slots k_accumulate folds into the buckets now (the others were traced ahead of the caller's Accumulate() calls)
};
struct QueueDev {
	float4* A[2]; float4* B[2]; float* T[2];
	uint32_t* N[2];          // [cap] the wide node a path's closest-hit walk starts at (the node holding the sphere it leaves from; written by k_shade, not read at bounce 0)
	float2* H;
	float4* SA; float4* SB; float* SL;
	uint32_t* SS;            // [cap] the wide node a shadow ray's walk starts at (the node holding the sphere it leaves from)
	uint32_t cap;
};
struct CountDev {            // zeroed at the start of every batch; index = bounce
	uint32_t* paths;         // [mb+1] paths entering bounce b
	uint32_t* shadow;        // [mb]   shadow rays queued at bounce b
	uint32_t* work_a;        // [mb]   work-fetch cursors of the traversal kernels
	uint32_t* work_b;        // [mb]
	unsigned long long* stats;  // [ST_COUNT] cumulative since reset_counters
};
// B2R_FLAG_REFERENCE_EXACT: the reference's per-tile stream bookkeeping. A stream = one sample of one 16x16 tile (256 slots,
// RayStream<256>); e = stream * 256 + slot indexes `key` / `next_idx`; `slot` and `act` are double-buffered like the path queue.
struct ExactDev {
	uint8_t* slot[2];     // [cap] slot of queue entry i inside its stream at this bounce (bounce 0: the pixel's ID)
	uint16_t* act[2];     // [cap / 256] active rays of each stream at this bounce (bounce 0: 256)
	uint8_t* key;         // [cap] 1 + material of the survivor that sat in (stream, slot) this bounce, 0 = none; cleared by k_stream_rank
	uint32_t* next_idx;   // [cap] its index in the next path queue
};
struct Params {
	SceneDev scene; FrameDev frame; QueueDev q; CountDev cnt; ExactDev ex;
	const BatchDev* batch;
	float* rad;   // RAD
	float* acc;   // ACC
	// [n_mat] {transmission.rgb, eta}, eta = 0 when max(transmission) == 0: read by the DIELECTRIC shading routines only (B2R_FLAG_DIELECTRIC).
	// A scene table, but kept here at the end rather than in SceneDev, so the parameter block of every other instantiation keeps its layout.
	const float4* mat_diel;
};

// ---------------------------------------------------------------------------------------------- small helpers
// tile-order pixel index -> pixel coordinates (Renderer.hpp:85-88,114-115)
B2R_HD void pixel_xy(uint32_t t, const FrameDev& fr, int32_t* x, int32_t* y) {
	const uint32_t tile = t >> 8, id = t & 255u;
	const uint32_t ty = div_by(tile, fr.h_tiles, fr.h_tiles_magic), tx = tile - ty * fr.h_tiles;
	*x = static_cast<int32_t>(tx * 16u + (id & 15u));
	*y = static_cast<int32_t>(ty * 16u + (id >> 4));
}

struct PathState { float ox, oy, oz, dx, dy, dz, tr, tg, tb, pdf; uint32_t pid; };

// primary ray of (slot, pixel t): Renderer.hpp:97-127. LENS: the thin-lens ray (camera_lens_ray, lens.radius > 0). Its lens sample is drawn
// from branch 2 * max_bounces of the pixel's seed range [seed, seed + 2 mb + 1): branches 2b (light sample) and 2b + 1 (BRDF continuation)
// of bounces b < mb use at most 2 mb - 1, so that stream is used by nothing else, and the camera jitter keeps its stream (branch 0).
template <bool LENS = false>
B2R_HD PathState primary_path(const FrameDev& fr, const CameraParams& cam, uint32_t acc, uint32_t slot, uint32_t t, const LensParams& lens = LensParams{0.0f, 0.0f}) {
	Pcg rng{hash_2d(acc, pixel_seed(t, fr.max_bounces))};
	const float s0 = rng.next_unit(), s1 = rng.next_unit();
	int32_t x, y; pixel_xy(t, fr, &x, &y);
	PathState s;
	if constexpr (LENS) {
		Pcg lr{hash_2d(acc, pixel_seed(t, fr.max_bounces) + 2u * fr.max_bounces)};
		const float u0 = lr.next_unit(), u1 = lr.next_unit();
		f3 o, d; camera_lens_ray(cam, x, y, s0, s1, lens, u0, u1, &o, &d);
		s.ox = o.x; s.oy = o.y; s.oz = o.z; s.dx = d.x; s.dy = d.y; s.dz = d.z;
	} else {
		const f3 d = camera_dir(cam, x, y, s0, s1);
		s.ox = cam.px; s.oy = cam.py; s.oz = cam.pz; s.dx = d.x; s.dy = d.y; s.dz = d.z;
	}
	s.tr = s.tg = s.tb = 1.0f; s.pdf = 0.0f; s.pid = (slot << 26) | t;
	return s;
}


// ---------------------------------------------------------------------------------------------- shading
struct Surface {
	f3 P; TangentQuat T; float n_dot_v; f3 albedo; bool emissive; int32_t mat; float r2; f3 v_local; float alpha;  // GGX: albedo holds F0; v_local / alpha are only set (and read) by the GGX closure
	bool inside; float4 diel; f3 P_in;  // DIELECTRIC only: N was flipped (the ray leaves the sphere), {transmission.rgb, eta} (eta = 0: not dielectric), hit - 1e-4 N
};
struct ShadowRay { f3 o, d; float tfar; f3 L; };

// Smooth dielectric (B2R_FLAG_DIELECTRIC, DESIGN §2): v = the direction towards the viewer in the local frame (N = +z, flipped against
// the ray), r = the ratio of the indices of refraction (1 / eta entering, eta leaving). With c = clamp(v.z, 0, 1) and s2 = r^2 (1 - c^2),
// s2 >= 1 is total internal reflection (F = 1, reflected whatever u0 is: next_unit can return 1.0, Q4); otherwise ct = sqrt(1 - s2) and F is
// the unpolarised Fresnel reflectance. u0 < F reflects into (-v.x, -v.y, c), else the ray refracts into (-r v.x, -r v.y, -ct). Only + - * / and
// sqrt, so host (-ffp-contract=off) and device (-fmad=false) agree bit for bit. Returns true for a reflection.
B2R_HD bool dielectric_scatter(f3 v, float r, float u0, f3* dir, float* F) {
	const float c = sel_min(sel_max(v.z, 0.0f), 1.0f);
	const float s2 = r * r * (1.0f - c * c);
	if (s2 >= 1.0f) { *F = 1.0f; *dir = f3{-v.x, -v.y, c}; return true; }
	const float ct = sqrtf(1.0f - s2);
	const float rs = (r * c - ct) / (r * c + ct), rp = (r * ct - c) / (r * ct + c);
	*F = (rs * rs + rp * rp) * 0.5f;
	const bool refl = u0 < *F;
	*dir = refl ? f3{-v.x, -v.y, c} : f3{-r * v.x, -r * v.y, -ct};
	return refl;
}

// closest-hit shader, Renderer.hpp:169-214. GGX = the reference's `#define BRDF 1` build (Renderer.hpp:70,207-213): the closure takes F0 and
// alpha = roughness^2 + (1 - roughness^2) * gloss_decay_table[bounce]; the reference never declares that table, it is all zeros here as in
// oracle/ref_renderer_build.sh's build of the reference itself. DIELECTRIC (B2R_FLAG_DIELECTRIC): also the material's dielectric data, whether
// the ray leaves the sphere, and the refracted ray's origin, 1e-4 behind the surface.
template <bool GGX = false, bool DIELECTRIC = false>
B2R_HD Surface shade_surface(const SceneDev& sc, const PathState& s, float depth, int32_t prim, const float4* mat_diel = nullptr) {
	const float4 sp = ld4(sc.prims + prim);
	const f3 D{s.dx, s.dy, s.dz};
	const f3 hp{s.ox + D.x * depth, s.oy + D.y * depth, s.oz + D.z * depth};
	f3 N = unit3(f3{hp.x - sp.x, hp.y - sp.y, hp.z - sp.z});
	const bool flip = dot3(N, D) >= 0.0f;
	if (flip) N = f3{-N.x, -N.y, -N.z};  // backface
	Surface sf;
	sf.T = tangent_frame(N);
	const f3 vl = frame_to_local(sf.T, f3{-D.x, -D.y, -D.z});
	sf.n_dot_v = vl.z;
	sf.P = f3{hp.x + N.x * 1e-4f, hp.y + N.y * 1e-4f, hp.z + N.z * 1e-4f};
	sf.mat = sc.prim_mat[prim];
	const float4 al = ld4(sc.mat_albedo + sf.mat);
	sf.albedo = f3{al.x, al.y, al.z}; sf.emissive = al.w != 0.0f; sf.r2 = sp.w;
	if (GGX) {
		const float4 fr = ld4(sc.mat_f0 + sf.mat);
		float alpha = fr.w; alpha *= alpha;
		sf.albedo = f3{fr.x, fr.y, fr.z}; sf.alpha = alpha + (1.0f - alpha) * 0.0f; sf.v_local = vl;  // Renderer.hpp:210-212
	}
	if (DIELECTRIC) {
		sf.diel = ld4(mat_diel + sf.mat); sf.inside = flip; sf.v_local = vl;
		sf.P_in = f3{hp.x - N.x * 1e-4f, hp.y - N.y * 1e-4f, hp.z - N.z * 1e-4f};
	}
	return sf;
}
template <bool DIELECTRIC> B2R_HD bool is_dielectric(const Surface& sf) { return DIELECTRIC && sf.diel.w != 0.0f; }
// next-event estimation, Renderer.hpp:249-298. Returns false when no shadow ray is produced; a dielectric surface (delta BSDF) never makes one.
template <bool GGX = false, bool DIELECTRIC = false>
B2R_HD bool shade_light_sample(const SceneDev& sc, const Surface& sf, const PathState& s, int32_t hit_prim,
                                                   uint32_t acc, uint32_t seed, uint32_t bounce, ShadowRay* out) {
	if (is_dielectric<DIELECTRIC>(sf)) return false;
	if (sc.n_lights == 0u) return false;  // undefined in the reference (Q15); defined here as "no light sampling"
	Pcg rng{hash_2d(acc, seed + bounce * 2u)};  // Q3
	const float u0 = rng.next_unit(), u1 = rng.next_unit();
	const uint32_t pick = rng.next_below(sc.n_lights);
	const float4 ls = ld4(sc.light_sphere + pick), le = ld4(sc.light_emit + pick);
	if (as_int(le.w) == hit_prim) return false;  // Q9: geometry index vs BVH-order index, as in the reference
	f3 wc{ls.x - sf.P.x, ls.y - sf.P.y, ls.z - sf.P.z};
	const float d2 = dot3(wc, wc);
	if (d2 <= ls.w) return false;
	const float dist = sqrtf(d2);
	wc = scale3(wc, 1.0f / dist);
	const float sin2 = ls.w / d2;
	const float n_dot_w = (2.0f * sf.T.w) * (wc.z * sf.T.w + wc.x * sf.T.y - sf.T.x * wc.y) - wc.z;  // Renderer.hpp:271
	if (n_dot_w < 0.0f && sin2 < n_dot_w * n_dot_w) return false;
	float ldist, lpdf;
	const f3 L = sample_sphere_cone(wc, sin2, dist, ls.w, u0, u1, &ldist, &lpdf);
	const f3 ll = frame_to_local(sf.T, L);
	if (ll.z < 0.0f) return false;
	f3 rad{le.x * s.tr, le.y * s.tg, le.z * s.tb};
	if (GGX) { const f3 e = ggx_eval(sf.albedo, sf.alpha, ll, sf.v_local); rad = f3{rad.x * e.x, rad.y * e.y, rad.z * e.z}; }  // Closure<GGX>::eval, DataStreams.hpp:189-195
	else {
		const float f = B2R_INV_PI * sel_max(0.0f, ll.z);  // Closure<Lambertian>::eval, DataStreams.hpp:169-172
		rad = f3{rad.x * (sf.albedo.x * f), rad.y * (sf.albedo.y * f), rad.z * (sf.albedo.z * f)};
	}
	lpdf *= sc.light_sel_pdf;
	const float bpdf = GGX ? 0.0f : B2R_INV_PI * sel_max(0.0f, ll.z);  // Closure<GGX>::pdf is `return 0.0f; //TODO` in the reference (:196-198)
	const float w = power_heuristic_over_f(lpdf, bpdf);
	rad = scale3(rad, w);
	if (sel_max(sel_max(rad.x, rad.y), rad.z) <= 0.0f) return false;
	out->o = sf.P; out->d = L; out->tfar = ldist; out->L = rad;
	return true;
}
// emissive-hit contribution, Renderer.hpp:319-353. DIELECTRIC: a path continued from a dielectric surface carries pdf = -1 (no light sample
// competes with a delta BSDF), and its MIS weight is 1.
template <bool DIELECTRIC = false>
B2R_HD f3 shade_emission(const SceneDev& sc, const Surface& sf, const PathState& s, float depth, uint32_t bounce, bool mis) {
	const float4 em = ld4(sc.mat_emission + sf.mat);
	if (!mis) return f3{s.tr * em.x, s.tg * em.y, s.tb * em.z};  // this repo's MIS-off (Q23)
	if (bounce == 0) return f3{em.x, em.y, em.z};
	if (DIELECTRIC && s.pdf < 0.0f) return f3{s.tr * em.x, s.tg * em.y, s.tb * em.z};
	const float d2 = depth * (depth + sf.n_dot_v * (2.0f * sqrtf(sf.r2))) + sf.r2;  // law of cosines, Renderer.hpp:331
	const float w = power_heuristic(s.pdf, sc.light_sel_pdf * sphere_light_pdf(sf.r2, d2));
	return f3{(s.tr * w) * em.x, (s.tg * w) * em.y, (s.tb * w) * em.z};
}
// BRDF sampling + Russian roulette, Renderer.hpp:359-403. Returns false when the path is terminated by roulette. A dielectric surface
// (DIELECTRIC) reflects or refracts by the stream's first float (dielectric_scatter; the second is unused, roulette keeps the third), a
// refraction scales the throughput by the transmission and leaves from P_in, and the path stores pdf = -1 (specular predecessor).
template <bool GGX = false, bool DIELECTRIC = false>
B2R_HD bool shade_continue(const Surface& sf, PathState* s, uint32_t acc, uint32_t seed, uint32_t bounce) {
	Pcg rng{hash_2d(acc, seed + bounce * 2u + 1u)};
	const float u0 = rng.next_unit(), u1 = rng.next_unit();
	f3 dl, est = sf.albedo, o = sf.P;
	const bool delta = is_dielectric<DIELECTRIC>(sf);
	if (delta) {
		float F;
		if (dielectric_scatter(sf.v_local, sf.inside ? sf.diel.w : 1.0f / sf.diel.w, u0, &dl, &F)) est = f3{1.0f, 1.0f, 1.0f};
		else { est = f3{sf.diel.x, sf.diel.y, sf.diel.z}; o = sf.P_in; }
	}
	else if (GGX) ggx_sample(sf.albedo, sf.alpha, sf.v_local, u0, u1, &dl, &est);  // Closure<GGX>::sample, DataStreams.hpp:199-218
	else dl = cosine_hemisphere(u0, u1);
	f3 thr{s->tr * est.x, s->tg * est.y, s->tb * est.z};
	const float q = 1.0f - sel_max(thr.x, sel_max(thr.y, thr.z));
	if (rng.next_unit() < q) return false;
	thr = scale3(thr, 1.0f / sel_max(FLT_EPSILON, 1.0f - q));
	const f3 dw = frame_to_world(sf.T, dl);
	s->ox = o.x; s->oy = o.y; s->oz = o.z; s->dx = dw.x; s->dy = dw.y; s->dz = dw.z;
	s->tr = thr.x; s->tg = thr.y; s->tb = thr.z;
	s->pdf = delta ? -1.0f : GGX ? 0.0f : B2R_INV_PI * sel_max(0.0f, dw.z);  // pdf of the world-space direction (Q10); Closure<GGX>::pdf returns 0
	return true;
}
// miss shader with ambient sky, Renderer.hpp:411-420 + Sky::operator(), Primitives.hpp:35-46
B2R_HD f3 shade_sky(const SceneDev& sc, const PathState& s) {
	const float u = sc.hdri_fw * (0.5f + B2R_INV_TWO_PI * atan2_poly(s.dz, s.dx));
	const float v = sc.hdri_fh * (0.5f - B2R_INV_PI * asin_poly(s.dy));
	const float4 tx = ldg4(sc.hdri + (static_cast<int32_t>(v) * sc.hdri_w + static_cast<int32_t>(u)));
	// Q14: all three channels are scaled by throughput.r
	return f3{s.tr * (tx.x * sc.ambient[0]), s.tr * (tx.y * sc.ambient[1]), s.tr * (tx.z * sc.ambient[2])};
}
// Adds up to two contributions, in this order, to the path's radiance at its pixel. Only one thread ever touches a given
// (sample, pixel) entry during a launch, so on the device the additions are issued as fire-and-forget reductions (RED.ADD.F32:
// same-address operations of one thread stay ordered, the result is the plain left-to-right float sum) and the warp does not
// wait for an HBM read-modify-write round trip.
B2R_HD void rad_add(float* rad, uint32_t npix, uint32_t pid, f3 a, f3 b, bool has_a = true, bool has_b = true) {
	const uint32_t slot = pid >> 26, t = pid & kPixMask;
	float* r = rad + static_cast<size_t>(slot) * 3u * npix + t;
#if defined(__CUDA_ARCH__)
	if (has_a) { atomicAdd(r, a.x); atomicAdd(r + npix, a.y); atomicAdd(r + 2u * npix, a.z); }
	if (has_b) { atomicAdd(r, b.x); atomicAdd(r + npix, b.y); atomicAdd(r + 2u * npix, b.z); }
#else
	if (has_a) { r[0] += a.x; r[npix] += a.y; r[2u * npix] += a.z; }
	if (has_b) { r[0] += b.x; r[npix] += b.y; r[2u * npix] += b.z; }
#endif
}
B2R_HD void rad_zero(float* rad, uint32_t npix, uint32_t pid) {
	const uint32_t slot = pid >> 26, t = pid & kPixMask;
	float* r = rad + static_cast<size_t>(slot) * 3u * npix + t;
	r[0] = 0.0f; r[npix] = 0.0f; r[2u * npix] = 0.0f;
}

// ---------------------------------------------------------------------------------------------- BVH traversal
// Per-lane traversal of the 4-wide tree, written as a resumable state machine: *_begin() arms a ray, *_step() visits ONE node
// and returns false when the ray is finished. The persistent kernels keep 32 such machines per warp and refill finished lanes
// with new rays, so a warp is not held up by its longest ray.
//
// Slot layout (b2r_host.h): A = {c.xyz, r2}, B = {h.x, h.y, link, h.z} — a box as centre + half extents for EVERY slot. A leaf slot
// holds the sphere itself in A (no leaf fetch) and in h the half extent of a cube that encloses every ray the float sphere tests
// could report as a hit (leaf_half_extent below), so all four slots of a node run ONE uniform slab pass and a sphere test is only
// paid for when the ray really passes the sphere's box within [0, best]. The centre/half form needs no per-axis min/max:
// t_centre = c*inv - o*inv (one FMA), t_half = h*|inv| (>= 0), near = t_centre - t_half, far = t_centre + t_half.
struct Ray { float ox, oy, oz, dx, dy, dz; };

constexpr float kSlabWiden = 1.0000008f;  // the exit distance is widened by ~7 ulp: rounding of the four operations per plane never rejects a box
// Per-ray set-up of the slab test, shared by TravBase::arm and k_intersect_packet: i = 1/d, n = -o/d, a = |1/d| per axis.
// Rule: an axis keeps n only while |1/d| * (|ox| + |oy| + |oz| + 2^64) <= 2^126; otherwise n is NaN, every term of that axis is NaN and drops
// out of fminf / fmaxf, and the axis leaves every box unconstrained — exactly what a zero component (0 * inf) always did. Why it is safe:
// - conservative: an unconstrained axis only accepts more boxes, and a box test never decides a result (the sphere tests do);
// - no overflow on a kept axis: |n| <= 2^126 and, for box centres |c| <= 2^64, |c/d| <= 2^126, so t_centre is finite; a half extent h
//   with |h/d| > FLT_MAX turns near into -inf and far into +inf, which only widens the box. Without the rule a finite 1/d with
//   |o/d| > FLT_MAX (d = 1e-38 from o = 400) made n = -inf, every exit distance -inf, and the BVH rejected every box brute force hits;
// - domain: box centres stay below 2^64 when sphere bounds and origins are below 2^61 (where |c - o|^2 is finite in the sphere tests); a
//   direction with a component of at least 2^-60 keeps that axis, so an empty slot (h = -1e30) is still rejected. A finite origin with
//   every |d| component below about 2^-61 (like d = 0, which did so before the rule) has no constrained axis: empty slots then pass and
//   their zero sphere at the world origin is tested under the id ~kEmptyLink — outside the domain above;
// - a non-finite origin makes the sum non-finite: all three axes are unconstrained and the walk tests every sphere, as brute force does
//   (the sphere tests then see NaN: closest misses, any hit reports occlusion, on both sides).
// Exact zeros, subnormals and finite components with an overflowing 1/d all come out as unconstrained axes. Once per ray, not per node.
constexpr float kSlabReach = 18446744073709551616.0f;  // 2^64
constexpr float kSlabRange = 8.50705917302346159e37f;  // 2^126, a factor 4 below FLT_MAX
B2R_HD void slab_setup(float ox, float oy, float oz, float dx, float dy, float dz, float* ix, float* iy, float* iz, float* nx, float* ny, float* nz,
                       float* ax, float* ay, float* az) {
	const float sx = 1.0f / dx, sy = 1.0f / dy, sz = 1.0f / dz;
	const float reach = ((fabsf(ox) + fabsf(oy)) + fabsf(oz)) + kSlabReach;   // NaN or inf for a non-finite origin
	const float nan = from_bits(0x7fc00000u);
	*ix = sx; *iy = sy; *iz = sz;
	*nx = fabsf(sx) * reach <= kSlabRange ? -(ox * sx) : nan;
	*ny = fabsf(sy) * reach <= kSlabRange ? -(oy * sy) : nan;
	*nz = fabsf(sz) * reach <= kSlabRange ? -(oz * sz) : nan;
	*ax = fabsf(sx); *ay = fabsf(sy); *az = fabsf(sz);
}
B2R_HD void slab(const float4 a, const float4 b, float ix, float iy, float iz, float nx, float ny, float nz, float ax, float ay, float az,
                 float limit, float* tnear, bool* hit) {
	// box tests never decide a result (they are conservative), so FMA is used freely; a NaN (0 * inf on an axis the ray is parallel
	// to) drops out of fminf / fmaxf, which leaves that axis unconstrained. (ax, ay, az) = |1/d|.
	const float cx = fma_rn(a.x, ix, nx), cy = fma_rn(a.y, iy, ny), cz = fma_rn(a.z, iz, nz);
	const float t0 = fmaxf(fmaxf(fmaxf(fma_rn(-b.x, ax, cx), fma_rn(-b.y, ay, cy)), fma_rn(-b.w, az, cz)), 0.0f);
	const float t1 = fminf(fminf(fminf(fma_rn(b.x, ax, cx), fma_rn(b.y, ay, cy)), fma_rn(b.w, az, cz)), limit);
	*tnear = t0; *hit = t0 <= t1 * kSlabWiden;
}
#define B2R_CSWAP(ka, la, kb, lb) { const bool sw = kb < ka; const uint32_t tk = sw ? kb : ka, tl = sw ? lb : la; kb = sw ? ka : kb; lb = sw ? la : lb; ka = tk; la = tl; }

// Traversal stacks hold one 32-bit word per entry: wide-node index in the high bits, and in the remaining `tn_bits` low bits the
// leading bits of the (non-negative) entry distance, truncated, i.e. a lower bound that still culls when the entry is popped.
// tn_bits = 32 - bits needed for a node index (16 at 100k spheres: 8 mantissa bits; 13 at 1M), chosen by the flattener. The storage is a policy: a plain array
// for whole-ray callers, shared memory with a local-memory overflow in the persistent kernels (a 64-entry per-thread array in
// local memory made the stack the largest L1/L2 client of the first version — more sectors than the nodes themselves).
constexpr uint32_t kMaxWideNodes = 1u << 22;  // leaves >= 10 bits for the distance
struct ArrayStack {
	uint32_t e[kTraversalStack]; int sp;
	B2R_HD void reset() { sp = 0; }
	B2R_HD void push(uint32_t v) { e[sp++] = v; }
	B2R_HD uint32_t pop() { return e[--sp]; }
	B2R_HD bool empty() const { return sp == 0; }
	B2R_HD void room() {}                    // called before the (up to three) pushes of a node visit
	B2R_HD bool refill() { return false; }   // called when the stack has run empty: entries brought back from a backing store
};
B2R_HD uint32_t pack_entry(uint32_t node, uint32_t tnear_bits, uint32_t tn_bits) { return (node << tn_bits) | (tnear_bits >> (31u - tn_bits)); }
B2R_HD float entry_tnear(uint32_t e, uint32_t tn_bits) { return from_bits((e & ((1u << tn_bits) - 1u)) << (31u - tn_bits)); }
B2R_HD uint32_t entry_node(uint32_t e, uint32_t tn_bits) { return e >> tn_bits; }

// Both per-lane walks can start at the BOTTOM of the tree and climb: a ray that leaves a point on a sphere starts at the wide node that
// holds that sphere's leaf slot (scene.leaf_node), searches that subtree, and once it has nothing left there moves up to the parent, searches
// the parent's other children (the child it came from, `skip`, is not entered again), and so on up to the root. The parent index a climb needs
// is fetched one climb ahead (`up`), so no step waits for it. A walk started at node 0 never climbs (`root != 0` guards it) and never reads
// parent[]: it is the plain walk from the root. Which boxes a climbing walk tests differs from a root walk only in the ancestors of the start
// node, whose own boxes it never tests: boxes are conservative and never decide a result, so a skipped box test can only lose culling, never a
// sphere test the result depends on (each walk's comment says why its result is unchanged).
constexpr uint32_t kNoNode = 0xffffffffu;
struct TravBase {
	float ox, oy, oz, dx, dy, dz;   // ray
	float ix, iy, iz, nx, ny, nz;   // 1/d and -o/d
	float ax, ay, az;               // |1/d| (the per-lane walks pass fabsf(i) to slab() instead: FFMA takes |R| as a free operand modifier, so these are not live in a walk)
	uint32_t node;
	uint32_t root, up, skip;        // climbing walks: top of the subtree searched so far, its parent, and the child of `root` already searched
	B2R_HD void arm(const Ray& r) {
		ox = r.ox; oy = r.oy; oz = r.oz; dx = r.dx; dy = r.dy; dz = r.dz;
		slab_setup(r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, &ix, &iy, &iz, &nx, &ny, &nz, &ax, &ay, &az);
		node = 0u;
	}
	B2R_HD void start_at(uint32_t start, const uint32_t* __restrict__ parent) {
		node = root = start; up = start != 0u ? ldg_u32(parent + start) : 0u; skip = kNoNode;  // (the root's parent entry is 0)
	}
	// nothing is left below `root`: move up one level (node = the parent, to be visited next). False once the root has been searched.
	B2R_HD bool climb(const uint32_t* __restrict__ parent) {
		if (root == 0u) return false;
		skip = root; root = up; node = up; up = ldg_u32(parent + up);
		return true;
	}
};
// node access: STAGED = the node's eight float4 were copied to shared memory by the warp (kernels); otherwise read-only LDG
template <bool STAGED> B2R_HD float4 node_f4(const float4* n, int i) { return STAGED ? n[i] : ldg4(n + i); }
B2R_HD int first_bit(uint32_t m) {
#if defined(__CUDA_ARCH__)
	return __ffs(static_cast<int>(m)) - 1;
#else
	return __builtin_ctz(m);
#endif
}

// Closest hit == brute force over all spheres (BVH.hpp:311-318): a candidate replaces the best when d < best, or d == best with
// a lower sphere index (the brute-force loop keeps the first of equal distances, BVH.hpp:265); a node or a leaf is culled only
// when its box is entered beyond the best distance. All four slots are slab-tested in one uniform pass; the leaf slots that passed
// are sphere-tested right away from the staged row (they can only shorten `best`), then the inner slots that passed are ordered by
// entry distance and re-checked against the possibly shorter `best` before they are pushed.
// Secondary rays climb (TravBase): k_shade queues, with every path it continues, the node that holds the sphere the path leaves from, and
// k_intersect_closest starts there; the walk climbs when its stack and backing store are empty. The result is still exact: the closest hit
// is the lexicographic minimum of (d, id) over the sphere tests made, which does not depend on the order they are made in; a sphere that
// holds the minimum lies inside every box on its path from the root (boxes are conservative) and entered no later than d <= best, so no
// cull rejects it wherever the walk starts; and a climbing walk only tests fewer boxes (the start node's ancestors'), never fewer spheres
// that could hold the minimum. A walk that climbs to the root has searched every subtree a root walk searches. Measured on C3's bounce-1
// rays (tests/hostcheck hc_closest_climb_stats, DESIGN §4): the node visits stay (13.0 -> 12.8: every ancestor is still searched), the
// pushes and pops of entries that the first nearby hit makes useless drop from 3.4 to 0.9 per ray.
template <class Stack>
struct TravClosestT : TravBase {
	float best; int32_t prim;
	bool tail = false;  // B2R_FLAG_REFERENCE_EXACT: this ray sits in the scalar tail of its tile's stream (BVH.hpp:270-286)
	Stack stack;
	// start: the node the walk begins at and climbs from; a walk from the root (start = 0) never reads `parent`, which may then be null
	B2R_HD void begin(const Ray& r, bool scalar_tail = false, uint32_t start = 0u, const uint32_t* __restrict__ parent = nullptr) {
		arm(r); start_at(start, parent); best = FLT_MAX; prim = -1; tail = scalar_tail; stack.reset();
	}
	template <bool COUNT, bool STAGED, uint32_t TNB = 0u>  // TNB != 0: the stack-entry split is a compile-time constant (immediate shifts)
	B2R_HD bool visit(const float4* n, uint32_t tn_bits_rt, const uint32_t* __restrict__ parent, uint32_t* c_sphere, uint32_t* c_box) {
		const uint32_t tn_bits = TNB ? TNB : tn_bits_rt;
		uint32_t key[4], link[4]; uint32_t leaves = 0u;
#pragma unroll
		for (int k = 0; k < 4; k++) {
			const float4 a = node_f4<STAGED>(n, 2 * k), b = node_f4<STAGED>(n, 2 * k + 1);
			const int32_t l = as_int(b.z);
			float tn; bool h; slab(a, b, ix, iy, iz, nx, ny, nz, fabsf(ix), fabsf(iy), fabsf(iz), best, &tn, &h);
			if (COUNT && l != kEmptyLink) (*c_box)++;
			key[k] = (h && l >= 0 && static_cast<uint32_t>(l) != skip) ? bits(tn) : 0xffffffffu; link[k] = static_cast<uint32_t>(l);
			leaves |= (h && l < 0) ? (1u << k) : 0u;  // an empty slot's box (h = -1e30) fails every constrained axis: never hit by a ray that keeps one (slab_setup)
		}
		while (leaves) {
			const int k = first_bit(leaves);
			leaves &= leaves - 1u;
			const float4 sp = node_f4<STAGED>(n, 2 * k); const int32_t id = ~as_int(node_f4<STAGED>(n, 2 * k + 1).z);
			float d; if (COUNT) (*c_sphere)++;
			const bool cand = tail ? sphere_hit_closest_scalar(sp.x, sp.y, sp.z, sp.w, ox, oy, oz, dx, dy, dz, &d) : sphere_hit_closest(sp.x, sp.y, sp.z, sp.w, ox, oy, oz, dx, dy, dz, &d);
			if (cand) {
				if (d < best || (d == best && id < prim)) { best = d; prim = id; }
			}
		}
		// sort the (entry distance, link) pairs; non-negative floats order like their bit patterns, misses (0xffffffff) last. (Moving only the
		// nearest child to the front — three exchanges instead of five, the others pushed as they come — was measured: 13.36 -> 13.54
		// node visits per ray on C3 and 1 % MORE kernel time, so the full sort stays.)
		B2R_CSWAP(key[0], link[0], key[1], link[1]); B2R_CSWAP(key[2], link[2], key[3], link[3]);
		B2R_CSWAP(key[0], link[0], key[2], link[2]); B2R_CSWAP(key[1], link[1], key[3], link[3]);
		B2R_CSWAP(key[1], link[1], key[2], link[2]);
		stack.room();
		// a miss key is a NaN pattern, so one ordered compare says "hit and still within the best distance"
		if (from_bits(key[3]) <= best) stack.push(pack_entry(link[3], key[3], tn_bits));
		if (from_bits(key[2]) <= best) stack.push(pack_entry(link[2], key[2], tn_bits));
		if (from_bits(key[1]) <= best) stack.push(pack_entry(link[1], key[1], tn_bits));
		if (from_bits(key[0]) <= best) { node = link[0]; return true; }
		for (;;) {
			while (!stack.empty()) {
				const uint32_t e = stack.pop();
				if (entry_tnear(e, tn_bits) <= best) { node = entry_node(e, tn_bits); return true; }
			}
			if (!stack.refill()) return climb(parent);  // false: walked the whole tree
		}
	}
	// (parent last and defaulted: a walk from the root never reads it)
	template <bool COUNT>
	B2R_HD bool step(const WideNode* __restrict__ wide, uint32_t tn_bits, uint32_t* c_sphere, uint32_t* c_box, const uint32_t* __restrict__ parent = nullptr) { return visit<COUNT, false>(reinterpret_cast<const float4*>(wide + node), tn_bits, parent, c_sphere, c_box); }
	template <bool COUNT, uint32_t TNB = 0u>
	B2R_HD bool step_staged(const float4* n, uint32_t tn_bits, const uint32_t* __restrict__ parent, uint32_t* c_sphere, uint32_t* c_box) { return visit<COUNT, true, TNB>(n, tn_bits, parent, c_sphere, c_box); }
};
// Any hit along [0, tfar) — Traverse_shadow semantics (BVH.hpp:290-305): an order-independent boolean. The nearest hit child is visited
// next, the others are pushed (in a dense scene the occluder is usually close to the origin — C3: every shadow ray is occluded; 12.4 -> 10.2
// node visits per ray); the first occluding leaf sphere ends the walk.
// The walk climbs (TravBase). A shadow ray leaves a point on a sphere, and in a dense scene its occluder is usually a neighbour of that
// sphere: a walk from the root spends ~8 of its 12-13 node visits descending to the origin's neighbourhood before it tests the first
// sphere. So k_intersect_shadow starts each ray at the wide node that holds its origin sphere's leaf slot (SS, written by k_shade from
// scene.leaf_node). Any-hit is an order-independent boolean over the same sphere tests, and a ray that reaches the root has visited
// exactly the nodes a root walk would have, so results are unchanged; measured on C3's shadow rays (tests/hostcheck hc_anyhit_local_stats):
// 12.3 -> 6.5 node visits per ray for the shadow rays of camera-ray hits, 13.1 -> 8.5 for those of later bounces.
template <class Stack>
struct TravAnyT : TravBase {
	float tfar; bool occluded;
	Stack stack;
	B2R_HD void begin(const Ray& r, float limit, uint32_t start, const uint32_t* __restrict__ parent) {
		arm(r); start_at(start, parent); tfar = limit; occluded = false; stack.reset();
	}
	template <bool COUNT, bool STAGED>
	B2R_HD bool visit(const float4* n, const uint32_t* __restrict__ parent, uint32_t* c_sphere, uint32_t* c_box) {
		uint32_t next = kNoNode, leaves = 0u; float next_tn = FLT_MAX;
		stack.room();
#pragma unroll
		for (int k = 0; k < 4; k++) {
			const float4 a = node_f4<STAGED>(n, 2 * k), b = node_f4<STAGED>(n, 2 * k + 1);
			const int32_t l = as_int(b.z);
			float tn; bool h; slab(a, b, ix, iy, iz, nx, ny, nz, fabsf(ix), fabsf(iy), fabsf(iz), tfar, &tn, &h);
			if (COUNT && l != kEmptyLink) (*c_box)++;
			if (h && l >= 0 && static_cast<uint32_t>(l) != skip) {
				const bool nearer = tn < next_tn;
				const uint32_t later = nearer ? next : static_cast<uint32_t>(l);
				if (later != kNoNode) stack.push(later);
				if (nearer) { next = static_cast<uint32_t>(l); next_tn = tn; }
			}
			leaves |= (h && l < 0) ? (1u << k) : 0u;  // leaf slots whose (inflated) box the ray passes within [0, tfar]
		}
		while (leaves) {
			const int k = first_bit(leaves);
			leaves &= leaves - 1u;
			const float4 sp = node_f4<STAGED>(n, 2 * k);
			if (COUNT) (*c_sphere)++;
			if (sphere_hit_any(sp.x, sp.y, sp.z, sp.w, ox, oy, oz, dx, dy, dz, tfar)) { occluded = true; return false; }
		}
		if (next == kNoNode && (!stack.empty() || stack.refill())) next = stack.pop();
		if (next != kNoNode) { node = next; return true; }
		return climb(parent);  // false: walked the whole tree without an occluder
	}
	template <bool COUNT>
	B2R_HD bool step(const WideNode* __restrict__ wide, const uint32_t* __restrict__ parent, uint32_t* c_sphere, uint32_t* c_box) { return visit<COUNT, false>(reinterpret_cast<const float4*>(wide + node), parent, c_sphere, c_box); }
	template <bool COUNT>
	B2R_HD bool step_staged(const float4* n, const uint32_t* __restrict__ parent, uint32_t* c_sphere, uint32_t* c_box) { return visit<COUNT, true>(n, parent, c_sphere, c_box); }
};
using TravClosest = TravClosestT<ArrayStack>;
using TravAny = TravAnyT<ArrayStack>;
// whole-ray wrappers (trace taps, host check). start: the node the walk begins at and climbs from; a walk from the root (start = 0) never
// reads `parent`, which may then be null
template <bool COUNT>
B2R_HD void traverse_closest(const WideNode* __restrict__ wide, uint32_t tn_bits, const Ray& r, float* best_out, int32_t* prim_out, uint32_t* c_sphere, uint32_t* c_box,
                             const uint32_t* __restrict__ parent = nullptr, uint32_t start = 0u, bool scalar_tail = false) {
	TravClosest t; t.begin(r, scalar_tail, start, parent);
	while (t.template step<COUNT>(wide, tn_bits, c_sphere, c_box, parent)) {}
	*best_out = t.best; *prim_out = t.prim;
}
template <bool COUNT>
B2R_HD bool traverse_any(const WideNode* __restrict__ wide, const Ray& r, float tfar, uint32_t* c_sphere, uint32_t* c_box, const uint32_t* __restrict__ parent = nullptr, uint32_t start = 0u) {
	TravAny t; t.begin(r, tfar, start, parent);
	while (t.template step<COUNT>(wide, parent, c_sphere, c_box)) {}
	return t.occluded;
}

// ------------------------------------------------------------------ slot boxes: build and refit (scene edit, Application.cpp:508-509)
// Leaf half extent. The closest hit is DEFINED as what the float sphere tests report (== the reference's brute force), and those tests
// are noisy: with t = c - o the discriminant b^2 - |t|^2 + r^2 cancels at the magnitude |t|^2, so a ray that passes the sphere at
// perpendicular distance p is reported as a hit whenever p^2 <= r^2 + E with E <= kHitNoise * |t|^2. Bound: the FMA form (BVH.hpp:252-260)
// makes 3 roundings of b (each <= u|t|, u = 2^-24) -> 2|b| * 3u|t| <= 6u|t|^2, 3 roundings of r^2 - |t|^2 -> 3u|t|^2, |d|^2 = 1 +- 4u
// -> 4u b^2; the dot-product form of the any-hit test (BVH.hpp:294-300) makes 5 + 1 + 5 + 2 roundings -> <= 18u|t|^2; the box test sees
// c and o separately, not t = fl(c - o): a shift of <= sqrt(3) u|t| -> < 4u|t|^2. 22u = 1.31e-6; kHitNoise rounds that up. A cube of half
// extent H = sqrt(r^2 + kHitNoise * D^2) around c therefore contains every ray either test can report, for every ray origin within
// distance D of c; D is taken over the scene's origin box (all sphere bounds, the camera, caller-supplied ray origins; b2r_host.h).
constexpr float kHitNoise = 1.5e-6f;
constexpr float kBoxPad = 4.0e-7f;  // outward padding, relative to |centre| + half extent + 1: covers the roundings of c -+ h below
B2R_HD float leaf_half_extent(const float4 s /*{c.xyz, r^2}*/, const OriginBox& ob) {
	const float ex = sel_max(fabsf(s.x - ob.lo[0]), fabsf(ob.hi[0] - s.x)), ey = sel_max(fabsf(s.y - ob.lo[1]), fabsf(ob.hi[1] - s.y)), ez = sel_max(fabsf(s.z - ob.lo[2]), fabsf(ob.hi[2] - s.z));
	const float far2 = (ex * ex + ey * ey + ez * ez) * 1.0001f;
	const float h = sqrtf(s.w + kHitNoise * far2);
	return h + (sel_max(fabsf(s.x), sel_max(fabsf(s.y), fabsf(s.z))) + h + 1.0f) * kBoxPad;
}
// The box of one inner slot, recomputed from the child wide node it links to: centre and half extents of the union of the child's
// slot boxes c -+ h (leaf slots included — their h is the inflated sphere extent), padded. The same routine fills the tree when it is
// built (flatten_bvh runs it level by level on the host), so a refit with unchanged spheres reproduces the built tree bit for bit.
B2R_HD void refit_child_box(const float4* __restrict__ child /*the 8 float4 of the linked wide node*/, float4* a_out, float4* b_out, int32_t link) {
	float lx = FLT_MAX, ly = FLT_MAX, lz = FLT_MAX, hx = -FLT_MAX, hy = -FLT_MAX, hz = -FLT_MAX;
	for (int j = 0; j < 4; j++) {
		const float4 ca = child[2 * j], cb = child[2 * j + 1];
		if (static_cast<int32_t>(bits(cb.z)) == kEmptyLink) continue;
		lx = sel_min(lx, ca.x - cb.x); ly = sel_min(ly, ca.y - cb.y); lz = sel_min(lz, ca.z - cb.w);
		hx = sel_max(hx, ca.x + cb.x); hy = sel_max(hy, ca.y + cb.y); hz = sel_max(hz, ca.z + cb.w);
	}
	const float cx = 0.5f * (lx + hx), cy = 0.5f * (ly + hy), cz = 0.5f * (lz + hz);
	float ex = sel_max(hx - cx, cx - lx), ey = sel_max(hy - cy, cy - ly), ez = sel_max(hz - cz, cz - lz);
	ex += (fabsf(cx) + ex + 1.0f) * kBoxPad; ey += (fabsf(cy) + ey + 1.0f) * kBoxPad; ez += (fabsf(cz) + ez + 1.0f) * kBoxPad;
	*a_out = make_float4(cx, cy, cz, 0.0f); *b_out = make_float4(ex, ey, from_bits(static_cast<uint32_t>(link)), ez);
}
// One slot of one wide node: leaf slots take the (moved) sphere and its inflated extent, inner slots the recomputed box. Levels are
// processed deepest first, so the child node read here is already final. `remap` (may be null = unchanged order) maps the BVH-order index a leaf
// held so far to the sphere's index in the new `prims` order (the reference re-sorts its prims on every rebuild, BVH.hpp:201-205, and
// hit indices must be indices into the current order: Q6 ties, Q9).
B2R_HD void refit_slot(float4* __restrict__ wide /*8 float4 per node*/, const float4* __restrict__ prims, const uint32_t* __restrict__ remap, const OriginBox& ob, uint32_t node, int k) {
	float4* slot = wide + static_cast<size_t>(node) * 8 + 2 * k;
	const int32_t link = static_cast<int32_t>(bits(slot[1].z));
	if (link == kEmptyLink) return;
	if (link < 0) {
		const uint32_t now = remap ? remap[~link] : static_cast<uint32_t>(~link);
		const float4 s = prims[now]; const float h = leaf_half_extent(s, ob);
		slot[0] = s; slot[1] = make_float4(h, h, from_bits(~now), h);
		return;
	}
	float4 a, b; refit_child_box(wide + static_cast<size_t>(link) * 8, &a, &b, link);
	slot[0] = a; slot[1] = b;
}
// 30-bit curve key of a sphere centre inside the sphere bounds [lo, hi] (10 bits per axis: the cell's Hilbert index; -DB2R_MORTON_ORDER = the Z-curve
// code it replaced, for A/B runs); shared by the GPU tree builds and their host twins
B2R_HD uint32_t morton_spread10(uint32_t v) { v &= 1023u; v = (v | (v << 16)) & 0x030000ffu; v = (v | (v << 8)) & 0x0300f00fu; v = (v | (v << 4)) & 0x030c30c3u; v = (v | (v << 2)) & 0x09249249u; return v; }
B2R_HD uint32_t morton_key(float cx, float cy, float cz, const float lo[3], const float scale[3]) {
	const float fx = (cx - lo[0]) * scale[0], fy = (cy - lo[1]) * scale[1], fz = (cz - lo[2]) * scale[2];
	const uint32_t qx = static_cast<uint32_t>(sel_min(sel_max(fx, 0.0f), 1023.0f)), qy = static_cast<uint32_t>(sel_min(sel_max(fy, 0.0f), 1023.0f)), qz = static_cast<uint32_t>(sel_min(sel_max(fz, 0.0f), 1023.0f));
#if defined(B2R_MORTON_ORDER)
	return (morton_spread10(qx) << 2) | (morton_spread10(qy) << 1) | morton_spread10(qz);
#else
	// Hilbert index of the cell (Skilling's transpose form, 10 bits per axis): unlike a Z curve, a run of consecutive cells is always a
	// connected, compact set, and the packed tree's nodes ARE runs of consecutive keys
	uint32_t x0 = qx, x1 = qy, x2 = qz;
	for (uint32_t q = 512u; q > 1u; q >>= 1) {
		const uint32_t m = q - 1u; uint32_t t;
		if (x0 & q) x0 ^= m;
		if (x1 & q) x0 ^= m; else { t = (x0 ^ x1) & m; x0 ^= t; x1 ^= t; }
		if (x2 & q) x0 ^= m; else { t = (x0 ^ x2) & m; x0 ^= t; x2 ^= t; }
	}
	x1 ^= x0; x2 ^= x1;
	uint32_t t = 0u;
	for (uint32_t q = 512u; q > 1u; q >>= 1) if (x2 & q) t ^= q - 1u;
	x0 ^= t; x1 ^= t; x2 ^= t;
	return (morton_spread10(x0) << 2) | (morton_spread10(x1) << 1) | morton_spread10(x2);
#endif
}
// ---- sweep build of the device tree (B2R_FLAG_GPU_SAH): arithmetic shared by k_sweep_* (b2r_device.cuh) and the host twin build_sweep_tree (b2r_host.cpp).
// The spheres stay in curve order; a node is a run [a, b) of that order, split where area(left) * count(left) + area(right) * count(right)
// is smallest (a surface-area-heuristic sweep along the curve instead of along three axes), the run with the largest box opened first
// until a node has four runs — the same greedy 2 -> 4 collapse flatten_bvh applies to a binary tree.
struct SweepItem { float lo0, lo1, lo2; uint32_t pos; float hi0, hi1, hi2; uint32_t flag; };  // a box + the segmented-scan bookkeeping (32 B)
B2R_HD SweepItem sweep_join(const SweepItem& a, const SweepItem& b) {  // segmented union, associative: an item that starts a segment forgets what is left of it
	if (b.flag) return b;
	SweepItem r;
	r.lo0 = sel_min(a.lo0, b.lo0); r.lo1 = sel_min(a.lo1, b.lo1); r.lo2 = sel_min(a.lo2, b.lo2);
	r.hi0 = sel_max(a.hi0, b.hi0); r.hi1 = sel_max(a.hi1, b.hi1); r.hi2 = sel_max(a.hi2, b.hi2);
	r.pos = a.pos; r.flag = a.flag;
	return r;
}
B2R_HD float sweep_area(const SweepItem& s) { const float ex = s.hi0 - s.lo0, ey = s.hi1 - s.lo1, ez = s.hi2 - s.lo2; return ex * ey + ey * ez + ez * ex; }
B2R_HD void sweep_sphere_box(const float4 s, SweepItem* it) {
	const float r = sqrtf(s.w);
	it->lo0 = s.x - r; it->lo1 = s.y - r; it->lo2 = s.z - r; it->hi0 = s.x + r; it->hi1 = s.y + r; it->hi2 = s.z + r; it->pos = 0u; it->flag = 0u;
}
// cost of cutting a run in front of position `pos`, packed so that an unsigned minimum picks the cheapest cut and, among equals, the first
B2R_HD unsigned long long sweep_key(float area_l, uint32_t n_l, float area_r, uint32_t n_r, uint32_t pos) {
	const float cost = area_l * static_cast<float>(n_l) + area_r * static_cast<float>(n_r);
	return (static_cast<unsigned long long>(bits(cost)) << 32) | pos;
}
struct SweepKids { uint32_t a[4], b[4], n; };  // the runs of one node while it is being opened (list order = slot order of flatten_bvh's collapse)
// one opening round: the run with the largest box among those holding two or more spheres is cut at its best position (cut_of[start of the
// run], area_of[start of the run]); the left part keeps its place in the list, the right part goes to the end. Returns the cut or 0 (none).
B2R_HD uint32_t sweep_open(SweepKids& K, const unsigned long long* cut_of, const float* area_of) {
	if (K.n >= 4u) return 0u;
	int pick = -1; float best = -1.0f;
	for (uint32_t k = 0; k < K.n; k++) if (K.b[k] - K.a[k] >= 2u) { const float ar = area_of[K.a[k]]; if (ar > best) { best = ar; pick = static_cast<int>(k); } }
	if (pick < 0) return 0u;
	const uint32_t pos = static_cast<uint32_t>(cut_of[K.a[pick]] & 0xffffffffull);
	K.a[K.n] = pos; K.b[K.n] = K.b[pick]; K.b[pick] = pos; K.n++;
	return pos;
}
// the four links of a finished node: runs of two or more spheres first (children child_first, child_first + 1, ... of the next level, their
// ranges returned), then single spheres (~index in the caller's sphere order), both in list order, then empty slots. Returns the child count.
B2R_HD uint32_t sweep_links(const SweepKids& K, const uint32_t* order, uint32_t child_first, int32_t link[4], uint32_t child_a[4], uint32_t child_b[4]) {
	uint32_t ni = 0u; int s = 0;
	for (uint32_t k = 0; k < K.n; k++) if (K.b[k] - K.a[k] >= 2u) { link[s++] = static_cast<int32_t>(child_first + ni); child_a[ni] = K.a[k]; child_b[ni] = K.b[k]; ni++; }
	for (uint32_t k = 0; k < K.n; k++) if (K.b[k] - K.a[k] == 1u) link[s++] = ~static_cast<int32_t>(order[K.a[k]]);
	for (; s < 4; s++) link[s] = kEmptyLink;
	return ni;
}
// ---- the three-axis variant (B2R_FLAG_GPU_SAH3): the same top-down sweep over three orders at once — the spheres sorted by centre x, y and z —
// every run being the same index range [a, b) of all three; a cut is (axis, position): the first position - a spheres of that axis' order go left.
B2R_HD uint32_t float_order_key(float f) { const uint32_t u = bits(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }  // unsigned order == float order
B2R_HD unsigned long long sweep_key3(float area_l, uint32_t n_l, float area_r, uint32_t n_r, uint32_t pos, uint32_t axis) {   // cheapest cost, then lowest position, then lowest axis
	const float cost = area_l * static_cast<float>(n_l) + area_r * static_cast<float>(n_r);
	return (static_cast<unsigned long long>(bits(cost)) << 32) | (pos << 2) | axis;
}
B2R_HD uint32_t sweep_open3(SweepKids& K, const unsigned long long* cut_of, const float* area_of, uint32_t* axis, uint32_t* run_a, uint32_t* run_b) {
	if (K.n >= 4u) return 0u;
	int pick = -1; float best = -1.0f;
	for (uint32_t k = 0; k < K.n; k++) if (K.b[k] - K.a[k] >= 2u) { const float ar = area_of[K.a[k]]; if (ar > best) { best = ar; pick = static_cast<int>(k); } }
	if (pick < 0) return 0u;
	const uint32_t low = static_cast<uint32_t>(cut_of[K.a[pick]] & 0xffffffffull), pos = low >> 2;
	*axis = low & 3u; *run_a = K.a[pick]; *run_b = K.b[pick];
	K.a[K.n] = pos; K.b[K.n] = K.b[pick]; K.b[pick] = pos; K.n++;
	return pos;
}
constexpr uint32_t kSweepMaxLevels = 20u;  // 3 stack entries per level must fit kTraversalStack; a deeper tree falls back to the packed one

B2R_HD void morton_scale(const float lo[3], const float hi[3], float scale[3]) { for (int k = 0; k < 3; k++) { const float e = hi[k] - lo[k]; scale[k] = e > 0.0f ? 1024.0f / e : 0.0f; } }
B2R_HD float slot_half_area(const float4 /*a*/, const float4 b) { return 4.0f * (b.x * b.y + b.y * b.w + b.w * b.x); }

}  // namespace b2r
