// lens_oracle.cpp — TEST HARNESS (compiled by tests/test_thin_lens.py, never part of libb2r.so).
//
// The CPU oracle (oracle/oracle.cpp, unchanged) with a thin lens restated from this repo's definition (b2r_math.h camera_lens_ray,
// b2r_set_lens; the reference has no lens, SURVEY Q22, so no reference result exists). The oracle is included whole; its renderer's
// per-tile loop calls generate_ray(c, ...) with a NON-const Ctx, so the overload declared below — an exact match that binds the non-const
// reference — is the one that loop calls, and it takes the lens branch for a context whose lens radius is > 0. The oracle's own
// generate_ray(const Ctx&, ...) stays the pinhole (R = 0, and every call through a const context).
#include <cstdint>
#include <map>
#include "oracle_math.hpp"

namespace {
struct Ctx;
static void generate_ray(Ctx& c, int32_t x, int32_t y, const float* samples, orc::V3* origin, orc::V3* dir);
}  // namespace

#include "oracle.cpp"

namespace {
struct Lens { float radius = 0.0f, focus = 1.0f; };
std::map<const Ctx*, Lens> g_lens;  // written by lo_set_lens between renders, only read while tiles run

// focus point P = v * (-F / z), lens point L = (r cos phi, r sin phi, 0) with r = R sqrt(u0), phi = 2 pi u1 (fast_sincos);
// origin = pos + orient * L, dir = normalize(orient * (P - L))
void generate_ray_lens(const Ctx& c, const Lens& lens, int32_t x, int32_t y, const float* samples, const float* lens_samples, V3* origin, V3* dir) {
	const V3 v{static_cast<float>(x) + samples[0] - c.half_width, static_cast<float>(y) + samples[1] - c.half_height, c.cam_z};
	const V3 P = v * (-lens.focus / c.cam_z);
	float sin_phi, cos_phi; fast_sincos(lens_samples[1] * kTwoPi, &sin_phi, &cos_phi);
	const float r = lens.radius * std::sqrt(lens_samples[0]);
	const V3 L{r * cos_phi, r * sin_phi, 0.0f};
	*origin = c.cam_pos + qrotate(c.cam_orient, L);
	*dir = normalize(qrotate(c.cam_orient, P - L));
}
// the camera ray of pixel (x, y), sample acc, for the pixel jitter `samples`: the lens sample is drawn from branch 2 * max_bounces of the
// pixel's seed range t * (2 mb + 1), which no light sample (2b) or BRDF continuation (2b + 1) uses
void camera_ray(const Ctx& c, int32_t x, int32_t y, uint32_t acc, const float* samples, V3* o, V3* d) {
	const auto it = g_lens.find(&c);
	if (it == g_lens.end() || !(it->second.radius > 0.0f)) { generate_ray(c, x, y, samples, o, d); return; }
	const uint32_t tile = static_cast<uint32_t>(y / kTileRoot) * c.h_tiles + static_cast<uint32_t>(x / kTileRoot);
	const uint32_t t = tile * kTileSize + static_cast<uint32_t>((y % kTileRoot) * kTileRoot + x % kTileRoot);
	const uint32_t seed = t * (c.max_bounces * 2u + 1u);
	uint32_t st = hash_2d(acc, seed + 2u * c.max_bounces);
	const float lens_samples[2] = {rand_unit_float(&st), rand_unit_float(&st)};
	generate_ray_lens(c, it->second, x, y, samples, lens_samples, o, d);
}
static void generate_ray(Ctx& c, int32_t x, int32_t y, const float* samples, V3* origin, V3* dir) {
	camera_ray(c, x, y, c.accumulations, samples, origin, dir);  // (the per-tile loop traces sample c.accumulations)
}
}  // namespace

extern "C" {
void lo_set_lens(Ctx* c, float radius, float focus) { g_lens[c] = Lens{radius, focus}; }
// one thin-lens camera ray for caller-supplied pixel and lens samples (the lens settings of lo_set_lens)
void lo_generate_lens_ray_at(const Ctx* c, int32_t x, int32_t y, const float samples[2], const float lens_samples[2], float out[6]) {
	V3 o, d; generate_ray_lens(*c, g_lens[c], x, y, samples, lens_samples, &o, &d);
	out[0] = o.x; out[1] = o.y; out[2] = o.z; out[3] = d.x; out[4] = d.y; out[5] = d.z;
}
// camera rays of sample acc for every pixel, tile order (orc_generate_rays with the lens)
void lo_generate_rays(const Ctx* c, uint32_t acc, float* out) {
	for (uint32_t tile = 0; tile < c->h_tiles * c->v_tiles; tile++) for (int ID = 0; ID < kTileSize; ID++) {
		const uint32_t t = tile * kTileSize + static_cast<uint32_t>(ID);
		const int32_t x = kTileRoot * static_cast<int32_t>(tile % c->h_tiles) + ID % kTileRoot, y = kTileRoot * static_cast<int32_t>(tile / c->h_tiles) + ID / kTileRoot;
		uint32_t st = hash_2d(acc, t * (c->max_bounces * 2u + 1u));
		const float cs[2] = {rand_unit_float(&st), rand_unit_float(&st)};
		V3 o, d; camera_ray(*c, x, y, acc, cs, &o, &d);
		float* p = out + static_cast<size_t>(t) * 6; p[0] = o.x; p[1] = o.y; p[2] = o.z; p[3] = d.x; p[4] = d.y; p[5] = d.z;
	}
}
}  // extern "C"
