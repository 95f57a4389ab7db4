// lens_taps.cpp — TEST HARNESS (compiled by tests/test_thin_lens.py, never part of libb2r.so): the kernels' camera routines
// (csrc/b2r_math.h camera_lens_ray, csrc/b2r_shade.h primary_path) on the host, for comparison with lens_oracle.cpp.
#include "b2r_shade.h"

using namespace b2r;

extern "C" {
void hc_lens_ray(const float cam11[11], int32_t x, int32_t y, const float samples[2], float radius, float focus, const float lens_samples[2], float out[6]) {
	const CameraParams cam{cam11[0], cam11[1], cam11[2], cam11[3], cam11[4], cam11[5], cam11[6], cam11[7], cam11[8], cam11[9], cam11[10]};
	f3 o, d; camera_lens_ray(cam, x, y, samples[0], samples[1], LensParams{radius, focus}, lens_samples[0], lens_samples[1], &o, &d);
	out[0] = o.x; out[1] = o.y; out[2] = o.z; out[3] = d.x; out[4] = d.y; out[5] = d.z;
}
// primary_path of every pixel of sample acc (tile order, out[t * 6 + {o.xyz, d.xyz}]), as k_generate / k_intersect_packet / k_bounce_brute
// make them: radius 0 takes the pinhole instantiation
void hc_primary_rays(const float cam11[11], uint32_t width, uint32_t height, uint32_t max_bounces, uint32_t acc, float radius, float focus, float* out) {
	FrameDev fr{};
	fr.cam = CameraParams{cam11[0], cam11[1], cam11[2], cam11[3], cam11[4], cam11[5], cam11[6], cam11[7], cam11[8], cam11[9], cam11[10]};
	fr.width = width; fr.height = height; fr.h_tiles = width / 16; fr.npix = width * height; fr.h_tiles_magic = magic_for(fr.h_tiles); fr.npix_magic = magic_for(fr.npix); fr.max_bounces = max_bounces;
	const LensParams lens{radius, focus};
	for (uint32_t t = 0; t < fr.npix; t++) {
		const PathState s = radius > 0.0f ? primary_path<true>(fr, fr.cam, acc, 0, t, lens) : primary_path(fr, fr.cam, acc, 0, t);
		float* o = out + static_cast<size_t>(t) * 6; o[0] = s.ox; o[1] = s.oy; o[2] = s.oz; o[3] = s.dx; o[4] = s.dy; o[5] = s.dz;
	}
}
}  // extern "C"
