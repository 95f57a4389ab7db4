// b2r_math.h — scalar device math of the path tracer (RNG, camera, tangent frames, light sampling, tonemap).
//
// Every function is host+device so the CUDA kernels (b2r_device.cuh) and the host-side scene code
// (b2r_host.cpp) share one definition. Arithmetic contract (DESIGN.md "Numerics"): IEEE binary32,
// round-to-nearest, no contraction — the library is compiled with `nvcc -fmad=false` / `g++ -ffp-contract=off`,
// and a fused multiply-add appears only where fma_rn() is written out (the closest-hit sphere test, which is
// where the reference uses FMA intrinsics, BVH.hpp:252-260; and box tests, which never decide a result).
// With that, each function below returns bit-identical results on sm_100a and on the host.
// file:line citations are into the reference (/root/reference) whose behaviour each function reproduces.
#pragma once
#include <stdint.h>
#include <float.h>
#include <math.h>
#include <string.h>

#if defined(__CUDACC__)
#define B2R_HD __host__ __device__ __forceinline__
#else
#define B2R_HD inline
#endif

namespace b2r {

struct f3 { float x, y, z; };
struct TangentQuat { float w, x, y; };  // z component is always 0 (Sampling.hpp:149-158)

B2R_HD uint32_t bits(float f) {
#if defined(__CUDA_ARCH__)
	return __float_as_uint(f);
#else
	uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}
B2R_HD float from_bits(uint32_t u) {
#if defined(__CUDA_ARCH__)
	return __uint_as_float(u);
#else
	float f; memcpy(&f, &u, 4); return f;
#endif
}
B2R_HD float fma_rn(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
	return __fmaf_rn(a, b, c);
#else
	return fmaf(a, b, c);
#endif
}
B2R_HD float round_even(float x) {
#if defined(__CUDA_ARCH__)
	return rintf(x);
#else
	return nearbyintf(x);
#endif
}
B2R_HD bool sign_set(float f) { return (bits(f) >> 31) != 0u; }
// select-style max/min: NaN and signed-zero behaviour of std::max/std::min/glm::max/glm::min
B2R_HD float sel_max(float a, float b) { return (a < b) ? b : a; }
B2R_HD float sel_min(float a, float b) { return (b < a) ? b : a; }

// ------------------------------------------------------------------ counter-based RNG (Random.hpp)
// One stream per (sample index, pixel seed + branch): state0 = hash_2d(acc, seed + branch) (Renderer.hpp:117,255,362)
B2R_HD uint32_t hash_2d(uint32_t x, uint32_t y) {  // Random.hpp:45-50
	const uint32_t m = 0x41c64e6du;
	uint32_t qx = m * ((x >> 1) ^ y), qy = m * ((y >> 1) ^ x);
	return m * (qx ^ (qy >> 3));
}
B2R_HD uint32_t hash_u32(uint32_t i) {  // Random.hpp:36-43
	i ^= i >> 16; i *= 0x21f0aaadu; i ^= i >> 15; i *= 0xd35a2d97u; i ^= i >> 15;
	return i ^ 0xe6fe3bebu;
}
struct Pcg {  // Random.hpp:10-29: output(previous state), then LCG step
	uint32_t state;
	B2R_HD uint32_t next_u32() {
		uint32_t v = state;
		state = v * 747796405u + 2891336453u;
		v = ((v >> ((v >> 28) + 4u)) ^ v) * 277803737u;
		return (v >> 22) ^ v;
	}
	B2R_HD float next_unit() {  // Random.hpp:5,26-29 — in [0,1], 1.0f reachable (Q4)
#if defined(__CUDA_ARCH__)
		return __uint2float_rn(next_u32()) * 0x1p-32f;
#else
		return static_cast<float>(next_u32()) * 0x1p-32f;
#endif
	}
	B2R_HD uint32_t next_below(uint32_t range) {  // Random.hpp:31-34
		uint32_t v = static_cast<uint32_t>(next_unit() * static_cast<float>(range));
		return v < range - 1u ? v : range - 1u;
	}
};
// pixel seed (Renderer.hpp:106-108, Q2): t = tile*256 + ID is the pixel's tile-order index
B2R_HD uint32_t pixel_seed(uint32_t t, uint32_t max_bounces) { return t * (max_bounces * 2u + 1u); }

// ------------------------------------------------------------------ small vector helpers (glm scalar semantics)
B2R_HD float dot3(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
B2R_HD f3 cross3(f3 a, f3 b) { return {a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y}; }
B2R_HD f3 scale3(f3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
B2R_HD f3 unit3(f3 v) { return scale3(v, 1.0f / sqrtf(dot3(v, v))); }  // glm::normalize = v * inversesqrt(dot)

// ------------------------------------------------------------------ camera (Camera.hpp)
struct CameraParams {  // View + Projection as generate_ray reads them (Camera.hpp:80-88)
	float px, py, pz;         // view.pos
	float qw, qx, qy, qz;     // view.orient
	float half_width, half_height, z, exposure;
};
// glm quat * vec3:  v + ((q.xyz × v) * w + q.xyz × (q.xyz × v)) * 2
B2R_HD f3 quat_rotate(float qw, float qx, float qy, float qz, f3 v) {
	f3 q{qx, qy, qz};
	f3 uv = cross3(q, v), uuv = cross3(q, uv);
	return {v.x + (uv.x * qw + uuv.x) * 2.0f, v.y + (uv.y * qw + uuv.y) * 2.0f, v.z + (uv.z * qw + uuv.z) * 2.0f};
}
B2R_HD f3 camera_dir(const CameraParams& c, int32_t x, int32_t y, float s0, float s1) {  // Camera.hpp:80-88 (pinhole, Q22)
	f3 v{static_cast<float>(x) + s0 - c.half_width, static_cast<float>(y) + s1 - c.half_height, c.z};
	return unit3(quat_rotate(c.qw, c.qx, c.qy, c.qz, v));
}
// Thin lens (not in the reference: Camera.hpp computes an aperture it never uses, Q22). radius R and focus distance F in scene units; F is
// measured along the forward axis, so the plane in focus is camera-space z = -F. radius 0 = pinhole: callers take camera_dir instead (this
// routine at R = 0 rounds differently: v is scaled by -F/z).
struct LensParams { float radius, focus; };
// pinhole part v as camera_dir; focus point P = v * (-F / z); lens point L = (r cos phi, r sin phi, 0), r = R sqrt(u0), phi = 2 pi u1;
// origin = pos + orient * L, dir = normalize(orient * (P - L)). Same order of operations in the test oracle's generate_ray_lens (tests/lenscheck/lens_oracle.cpp).
B2R_HD void camera_lens_ray(const CameraParams& c, int32_t x, int32_t y, float s0, float s1, const LensParams& lens, float u0, float u1, f3* origin, f3* dir);
// glm::quatLookAt(normalize(forward), {0,1,0}) (Camera.hpp:47-50): RH basis {right, up', -dir} -> quat_cast
B2R_HD void look_at_quat(f3 forward, float out_wxyz[4]) {
	f3 d = unit3(forward);
	f3 back{-d.x, -d.y, -d.z};
	f3 r = cross3(f3{0.0f, 1.0f, 0.0f}, back);
	f3 right = scale3(r, 1.0f / sqrtf(sel_max(0.00001f, dot3(r, r))));
	f3 up = cross3(back, right);
	// trace-based branch selection of glm::quat_cast on the column-major 3x3 {right, up, back}
	float tw = right.x + up.y + back.z, tx = right.x - up.y - back.z, ty = up.y - right.x - back.z, tz = back.z - right.x - up.y;
	int sel = 0; float big = tw;
	if (tx > big) { big = tx; sel = 1; }
	if (ty > big) { big = ty; sel = 2; }
	if (tz > big) { big = tz; sel = 3; }
	float v = sqrtf(big + 1.0f) * 0.5f, m = 0.25f / v;
	float a = (up.z - back.y) * m, b = (back.x - right.z) * m, c = (right.y - up.x) * m;     // antisymmetric parts
	float sxy = (right.y + up.x) * m, sxz = (back.x + right.z) * m, syz = (up.z + back.y) * m; // symmetric parts
	if (sel == 0) { out_wxyz[0] = v; out_wxyz[1] = a; out_wxyz[2] = b; out_wxyz[3] = c; }
	else if (sel == 1) { out_wxyz[0] = a; out_wxyz[1] = v; out_wxyz[2] = sxy; out_wxyz[3] = sxz; }
	else if (sel == 2) { out_wxyz[0] = b; out_wxyz[1] = sxy; out_wxyz[2] = v; out_wxyz[3] = syz; }
	else { out_wxyz[0] = c; out_wxyz[1] = sxz; out_wxyz[2] = syz; out_wxyz[3] = v; }
}

// ------------------------------------------------------------------ trig approximations (VectorMath.hpp:625-662)
#define B2R_PI 3.14159265358979323846264338327950288f
#define B2R_TWO_PI 6.28318530717958647692528676655900576f
#define B2R_HALF_PI 1.57079632679489661923132169163975144f
#define B2R_INV_PI 0.318309886183790671537767526745028724f
#define B2R_INV_TWO_PI 0.159154943091895335768883763372514362f

B2R_HD void sincos_poly(float x, float* s_out, float* c_out) {  // fast_sincos, VectorMath.hpp:644-662
	const float q = round_even(x * B2R_INV_PI);
	const uint32_t flip = static_cast<uint32_t>(static_cast<int32_t>(q)) << 31;  // odd multiple of pi -> negate
	x += q * (-0.78515625f * 4.0f);                       // 4-step Cody-Waite reduction of x - q*pi
	x += q * (-0.00024187564849853515625f * 4.0f);
	x += q * (-3.7747668102383613586e-08f * 4.0f);
	x += q * (-1.2816720341285448015e-12f * 4.0f);
	x = B2R_HALF_PI - (B2R_HALF_PI - x);
	const float x2 = x * x;
	x = from_bits(bits(x) ^ flip);
	float s = 2.6083159809786593541503e-06f, c = -2.71811842367242206819355e-07f;
	s = s * x2 - 0.0001981069071916863322258f;  c = c * x2 + 2.47990446951007470488548e-05f;
	s = s * x2 + 0.00833307858556509017944336f; c = c * x2 - 0.00138888787478208541870117f;
	s = s * x2 - 0.166666597127914428710938f;   c = c * x2 + 0.0416666641831398010253906f;
	s = x2 * (s * x) + x;                       c = c * x2 - 0.5f; c = c * x2 + 1.0f;
	c = from_bits(bits(c) ^ flip);
	if (from_bits(bits(s) & 0x7fffffffu) > 1.0f) s = 0.0f;
	if (from_bits(bits(c) & 0x7fffffffu) > 1.0f) c = 0.0f;
	*s_out = s; *c_out = c;
}
B2R_HD void camera_lens_ray(const CameraParams& c, int32_t x, int32_t y, float s0, float s1, const LensParams& lens, float u0, float u1, f3* origin, f3* dir) {
	const f3 v{static_cast<float>(x) + s0 - c.half_width, static_cast<float>(y) + s1 - c.half_height, c.z};
	const f3 P = scale3(v, -lens.focus / c.z);
	float sn, cs; sincos_poly(u1 * B2R_TWO_PI, &sn, &cs);
	const float r = lens.radius * sqrtf(u0);
	const f3 L{r * cs, r * sn, 0.0f};
	const f3 lw = quat_rotate(c.qw, c.qx, c.qy, c.qz, L);
	*origin = f3{c.px + lw.x, c.py + lw.y, c.pz + lw.z};
	*dir = unit3(quat_rotate(c.qw, c.qx, c.qy, c.qz, f3{P.x - L.x, P.y - L.y, P.z - L.z}));
}
B2R_HD float asin_poly(float x) {  // fast_asin, VectorMath.hpp:625-630
	float f = from_bits(bits(x) & 0x7fffffffu);
	f = (f < 1.0f) ? 1.0f - (1.0f - f) : 1.0f;
	f = B2R_HALF_PI - sqrtf(1.0f - f) * (1.5707963267f + f * (-0.213300989f + f * (0.077980478f + f * -0.02164095f)));
	return from_bits((bits(f) & 0x7fffffffu) | (bits(x) & 0x80000000u));
}
B2R_HD float atan2_poly(float y, float x) {  // fast_atan2, VectorMath.hpp:632-642
	const float a = from_bits(bits(x) & 0x7fffffffu), b = from_bits(bits(y) & 0x7fffffffu);
	const float lo = sel_min(a, b), hi = sel_max(a, b);
	float k = hi == 0.0f ? 0.0f : lo / hi;
	k = 1.0f - (1.0f - k);
	const float k2 = k * k;
	float r = k * (0.43157974f * k2 + 1.0f) / ((0.05831938f * k2 + 0.76443945f) * k2 + 1.0f);
	if (b > a) r = B2R_HALF_PI - r;
	if (x < 0.0f) r = B2R_PI - r;
	return from_bits((bits(r) & 0x7fffffffu) | (bits(y) & 0x80000000u));
}

// ------------------------------------------------------------------ tangent frames and sampling (Sampling.hpp)
B2R_HD f3 sphere_coords(float phi_turns, float sin_t, float cos_t) {  // spherical_to_cartesian, Sampling.hpp:77-84
	float sp, cp; sincos_poly(phi_turns * B2R_TWO_PI, &sp, &cp);
	return {sin_t * cp, sin_t * sp, cos_t};
}
B2R_HD f3 cosine_hemisphere(float u0, float u1) {  // hemisphere, Sampling.hpp:92-94
	return sphere_coords(u1, sqrtf(u0), sqrtf(sel_max(0.0f, 1.0f - u0)));
}
B2R_HD TangentQuat tangent_frame(f3 n) {  // tangent_space, Sampling.hpp:150-159 (Frisvad quaternion; z == 0)
	if (n.z < -1.0f + FLT_EPSILON) return {0.0f, 0.0f, 1.0f};
	float s = sqrtf(2.0f * (n.z + 1.0f)), inv = 1.0f / s;
	return {s * 0.5f, -n.y * inv, n.x * inv};
}
B2R_HD f3 frame_to_local(TangentQuat t, f3 v) {  // to_local, Sampling.hpp:161-169
	float k = 2.0f * (v.z * t.w + v.x * t.y - t.x * v.y);
	return {v.x - t.y * k, v.y + t.x * k, k * t.w - v.z};
}
B2R_HD f3 frame_to_world(TangentQuat t, f3 v) {  // to_world, Sampling.hpp:171-179
	float k = 2.0f * (v.z * t.w - v.x * t.y + t.x * v.y);
	return {v.x + t.y * k, v.y - t.x * k, k * t.w - v.z};
}
B2R_HD void branchless_onb(f3 n, f3* u, f3* v) {  // orthonormal_basis, Sampling.hpp:116-131 (sign-bit variant)
	const uint32_t sg = bits(n.z) & 0x80000000u;
	const float s = from_bits(0x3f800000u ^ sg);
	const float z = -1.0f / (s + n.z);
	const float snx = from_bits(sg ^ bits(n.x));
	const float nyz = n.y * z;
	const float t = n.x * nyz;
	*u = f3{1.0f + (snx * n.x) * z, from_bits(sg ^ bits(t)), -snx};
	*v = f3{t, s + nyz * n.y, -n.y};
}
B2R_HD float cone_pdf(float cos_max) { return B2R_INV_TWO_PI / sel_max(1e-6f, 1.0f - cos_max); }  // Sampling.hpp:192-194
B2R_HD float sphere_light_pdf(float r2, float d2) {  // spherePdf, Sampling.hpp:196-200
	float s2 = r2 / d2;
	return cone_pdf(sqrtf(sel_max(0.0f, 1.0f - s2)));
}
// sample_direction_to_sphere, Sampling.hpp:220-239. wc: unit vector to the light centre.
B2R_HD f3 sample_sphere_cone(f3 wc, float sin2_max, float center_dist, float r2, float u0, float u1, float* dist_out, float* pdf_out) {
	const float cos_max = sqrtf(sel_max(0.0f, 1.0f - sin2_max));
	*pdf_out = cone_pdf(cos_max);
	const bool small_angle = sin2_max < 0.00068523f;  // Taylor branch below ~1.5 degrees
	float cos_t = 1.0f - u0 * (1.0f - cos_max);
	float sin_t = sqrtf(sin2_max * u0);
	const float src = small_angle ? sin_t : cos_t;
	const float other = sqrtf(sel_max(0.0f, 1.0f - src * src));
	cos_t = small_angle ? other : cos_t;
	sin_t = small_angle ? sin_t : other;
	const float h = center_dist * sin_t;
	*dist_out = center_dist * cos_t - sqrtf(sel_max(0.0f, r2 - h * h)) - 1e-5f;
	const f3 l = sphere_coords(u1, sin_t, cos_t);
	f3 bx, by; branchless_onb(wc, &bx, &by);
	return {bx.x * l.x + by.x * l.y + wc.x * l.z, bx.y * l.x + by.y * l.y + wc.y * l.z, bx.z * l.x + by.z * l.y + wc.z * l.z};
}
// ---- GGX closure (the reference's `#define BRDF 1` build: Closure<ClosureType::GGX>, DataStreams.hpp:184-219; Sampling.hpp:102-104,249-309)
B2R_HD float lerp_glm(float a, float b, float t) { return a * (1.0f - t) + b * t; }  // glm::mix(x, y, a) = x * (1 - a) + y * a
B2R_HD f3 ggx_visible_normal(f3 v_local, float alpha, float u0, float u1) {  // distribution_visible_normals, Sampling.hpp:253-270
	const f3 V = unit3(f3{alpha * v_local.x, alpha * v_local.y, v_local.z});
	float sn, cs; sincos_poly(u1 * B2R_TWO_PI, &sn, &cs);  // disk(u, v) = polar_to_cartesian(v, sqrt(u)), :85-91,102-104
	const float rho = sqrtf(u0);
	const float sx = rho * cs; float sy = rho * sn;
	const float t = 1.0f - sx * sx;
	sy = lerp_glm(sqrtf(t), sy, V.z * 0.5f + 0.5f);
	f3 X, Y; branchless_onb(V, &X, &Y);
	const float hz = sqrtf(sel_max(0.0f, t - sy * sy));
	const f3 H{(X.x * sx + Y.x * sy) + V.x * hz, (X.y * sx + Y.y * sy) + V.y * hz, (X.z * sx + Y.z * sy) + V.z * hz};
	return unit3(f3{alpha * H.x, alpha * H.y, sel_max(0.0f, H.z)});
}
B2R_HD f3 ggx_fresnel(f3 f0, float h_dot_v) {  // Fresnel, Sampling.hpp:272-275
	float c = 1.0f - h_dot_v; c = c < 0.0f ? 0.0f : (1.0f < c ? 1.0f : c);  // std::clamp
	float a = c * c; a *= a; a = c * a;  // pow5
	return f3{f0.x * (1.0f - a) + 1.0f * a, f0.y * (1.0f - a) + 1.0f * a, f0.z * (1.0f - a) + 1.0f * a};
}
B2R_HD float ggx_ndf(float alpha2, float n_dot_h2) { const float t = (1.0f + (alpha2 - 1.0f) * n_dot_h2); return alpha2 / (B2R_PI * t * t); }  // GGX_D, :278-281
B2R_HD float ggx_g2_lagarde(float alpha2, float n_dot_l, float n_dot_v) {  // Smith_G2_Height_Correlated_GGX_Lagarde, :287-291
	const float a = n_dot_v * sqrtf(alpha2 + n_dot_l * (n_dot_l - alpha2 * n_dot_l));
	const float b = n_dot_l * sqrtf(alpha2 + n_dot_v * (n_dot_v - alpha2 * n_dot_v));
	return 0.5f / (a + b);
}
B2R_HD f3 ggx_microfacet_brdf(f3 f0, float alpha, float n_dot_v, float n_dot_l, float n_dot_h, float h_dot_v) {  // microfacet_brdf, :293-296
	const float alpha2 = alpha * alpha;
	return scale3(ggx_fresnel(f0, h_dot_v), n_dot_l * ggx_ndf(sel_max(0.00001f, alpha2), n_dot_h * n_dot_h) * ggx_g2_lagarde(alpha2, n_dot_l, n_dot_v));
}
B2R_HD float ggx_g1(float alpha2, float n_dot_s2) { return 2.0f / (1.0f + sqrtf(((alpha2 * (1.0f - n_dot_s2)) + n_dot_s2) / n_dot_s2)); }  // G1_GGX, :297-299
B2R_HD f3 ggx_vndf_estimator(f3 f0, float alpha, float n_dot_v, float n_dot_l, float h_dot_v) {  // vndf_estimator, :301-309
	const float alpha2 = alpha * alpha;
	const float g1v = ggx_g1(alpha2, n_dot_v * n_dot_v), g1l = ggx_g1(alpha2, n_dot_l * n_dot_l);
	return scale3(ggx_fresnel(f0, h_dot_v), g1l / (g1v + g1l - g1v * g1l));
}
B2R_HD f3 ggx_eval(f3 f0, float alpha, f3 l_local, f3 v_local) {  // Closure<GGX>::eval, DataStreams.hpp:189-195
	const float n_dot_l = sel_max(0.0f, l_local.z), n_dot_v = sel_max(0.0f, v_local.z);
	const f3 hn = unit3(f3{l_local.x + v_local.x, l_local.y + v_local.y, l_local.z + v_local.z});
	return ggx_microfacet_brdf(f0, alpha, n_dot_v, n_dot_l, sel_max(0.0f, hn.z), sel_max(0.0f, dot3(hn, v_local)));
}
B2R_HD void ggx_sample(f3 f0, float alpha, f3 v_local, float u0, float u1, f3* dir, f3* estimator) {  // Closure<GGX>::sample, DataStreams.hpp:199-218
	const float n_dot_v = sel_max(0.0f, v_local.z);
	float h_dot_v;
	if (alpha == 0.0f) { *dir = f3{-v_local.x, -v_local.y, v_local.z}; h_dot_v = n_dot_v; }
	else {
		const f3 h = ggx_visible_normal(v_local, alpha, u0, u1);
		h_dot_v = dot3(h, v_local);
		const float k = 2.0f * h_dot_v;
		*dir = f3{k * h.x - v_local.x, k * h.y - v_local.y, k * h.z - v_local.z};
		h_dot_v = sel_max(0.0f, h_dot_v);
	}
	*estimator = ggx_vndf_estimator(f0, alpha, n_dot_v, sel_max(0.0f, dir->z), h_dot_v);
}
B2R_HD float power_heuristic(float f, float g) { float f2 = f * f; return f2 / sel_max(1e-6f, f2 + g * g); }  // Sampling.hpp:241-244
B2R_HD float power_heuristic_over_f(float f, float g) { return f / sel_max(1e-6f, f * f + g * g); }         // Sampling.hpp:245-247

// ------------------------------------------------------------------ sphere tests (BVH.hpp:236-305)
// Closest hit, one lane of the SIMD block BVH.hpp:251-267: returns the candidate distance, or a negative number /
// NaN-free sentinel when the lane's store mask is clear. sphere = {cx, cy, cz, r^2}.
// The part of the test that depends only on (sphere, ray origin): t = c - o and r^2 - |t|^2 in the reference's FMA order.
// Camera rays share one origin, so the bounce-0 kernel evaluates this once per sphere instead of once per ray.
struct SpherePre { float tx, ty, tz, disc0; };
B2R_HD SpherePre sphere_prepare(float cx, float cy, float cz, float r2, float ox, float oy, float oz) {
	SpherePre p; p.tx = cx - ox; p.ty = cy - oy; p.tz = cz - oz;
	p.disc0 = fma_rn(-p.tz, p.tz, fma_rn(-p.ty, p.ty, fma_rn(-p.tx, p.tx, r2)));
	return p;
}
B2R_HD bool sphere_hit_prepared(const SpherePre& p, float dx, float dy, float dz, float* dist_out) {
	const float b = fma_rn(dz, p.tz, fma_rn(dy, p.ty, dx * p.tx));
	const float disc = fma_rn(b, b, p.disc0);
	// The reference takes the square root unconditionally and masks afterwards (:262-265): a negative discriminant gives
	// NaN (fails the ordered compare) and -0 keeps its sign bit (masked out). Both are exactly "bit pattern above +inf",
	// so the root is only evaluated for discriminants in [+0, +inf].
	if (bits(disc) > 0x7f800000u) return false;
	const float root = sqrtf(disc);
	float d = b - root;
	if (sign_set(d)) d = b + root;  // blendv on the sign bit (:264)
	*dist_out = d;
	return !sign_set(d);            // NaN/inf distances fail the caller's `d < tfar`
}
B2R_HD bool sphere_hit_closest(float cx, float cy, float cz, float r2, float ox, float oy, float oz, float dx, float dy, float dz, float* dist_out) {
	return sphere_hit_prepared(sphere_prepare(cx, cy, cz, r2, ox, oy, oz), dx, dy, dz, dist_out);
}
// The scalar tail of the same loop, BVH.hpp:270-286 (no FMA; accumulation order x, y, z): the reference runs it for the last
// `active % 8` rays of a tile's stream. Only B2R_FLAG_REFERENCE_EXACT uses it. Updates (best, prim) exactly as the reference does.
B2R_HD void sphere_closest_scalar_update(float cx, float cy, float cz, float r2, int32_t id, float ox, float oy, float oz, float dx, float dy, float dz, float* best, int32_t* prim) {
	float b = 0.0f, disc = r2;
	float t = cx - ox; b += dx * t; disc -= t * t;
	t = cy - oy; b += dy * t; disc -= t * t;
	t = cz - oz; b += dz * t; disc -= t * t;
	disc += b * b;
	if (disc < 0.0f) return;
	disc = sqrtf(disc);
	const float dist = (b >= disc) ? b - disc : b + disc;
	if (dist < 0.0f || dist >= *best) return;
	*best = dist; *prim = id;
}
// the same formula as a candidate test (for the BVH traversal, where spheres are not met in index order): distance if the scalar
// tail would consider this sphere at all (discriminant >= 0 and distance >= 0); the caller applies `d < best`, ties to the lower index
B2R_HD bool sphere_hit_closest_scalar(float cx, float cy, float cz, float r2, float ox, float oy, float oz, float dx, float dy, float dz, float* dist_out) {
	float b = 0.0f, disc = r2;
	float t = cx - ox; b += dx * t; disc -= t * t;
	t = cy - oy; b += dy * t; disc -= t * t;
	t = cz - oz; b += dz * t; disc -= t * t;
	disc += b * b;
	if (disc < 0.0f) return false;
	disc = sqrtf(disc);
	const float dist = (b >= disc) ? b - disc : b + disc;
	*dist_out = dist;
	return !(dist < 0.0f);
}
// Any hit along [0, tfar): BVH.hpp:294-300 (glm dot products, no FMA)
B2R_HD bool sphere_hit_any(float cx, float cy, float cz, float r2, float ox, float oy, float oz, float dx, float dy, float dz, float tfar) {
	f3 p{cx - ox, cy - oy, cz - oz};
	float b = dot3(f3{dx, dy, dz}, p);
	float disc = b * b - dot3(p, p) + r2;
	if (disc < 0.0f) return false;
	disc = sqrtf(disc);
	float d = (b >= disc) ? b - disc : b + disc;
	return !(d < 0.0f || d >= tfar);
}

// ------------------------------------------------------------------ resolve (Renderer.hpp:436-478, Color.hpp:47-73)
B2R_HD float lane_min(float a, float b) { return (a < b) ? a : b; }  // _mm256_min_ps / _mm256_max_ps operand semantics
B2R_HD float lane_max(float a, float b) { return (a > b) ? a : b; }
B2R_HD float median_of_3(float a, float b, float c) { return lane_max(lane_min(a, b), lane_min(lane_max(a, b), c)); }  // Sampling.hpp:8-12
B2R_HD float median_of_5(float a, float b, float c, float d, float e) {  // Sampling.hpp:13-21
	return median_of_3(lane_max(lane_min(a, b), lane_min(c, d)), lane_min(lane_max(a, b), lane_max(c, d)), e);
}
// median of 8 (this repo's even-K definition: mean of the two middle order statistics) with Batcher's 19 compare-exchanges in
// registers; each exchange outputs a permutation of its inputs, so the result equals sorting the eight values.
#define B2R_CE(a, b) { const bool sw_ = b < a; const float lo_ = sw_ ? b : a; b = sw_ ? a : b; a = lo_; }
B2R_HD float median_of_8(float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7) {
	B2R_CE(v0, v1); B2R_CE(v2, v3); B2R_CE(v4, v5); B2R_CE(v6, v7);
	B2R_CE(v0, v2); B2R_CE(v1, v3); B2R_CE(v4, v6); B2R_CE(v5, v7);
	B2R_CE(v1, v2); B2R_CE(v5, v6);
	B2R_CE(v0, v4); B2R_CE(v1, v5); B2R_CE(v2, v6); B2R_CE(v3, v7);
	B2R_CE(v2, v4); B2R_CE(v3, v5);
	B2R_CE(v1, v2); B2R_CE(v3, v4); B2R_CE(v5, v6);
	return (v3 + v4) * 0.5f;
}
B2R_HD float aces_curve(float x) { return (x * (x + 0.0245786f) - 0.000090537f) / (x * (0.983729f * x + 0.4329510f) + 0.238081f); }  // Color.hpp:47-49
B2R_HD void aces_tonemap(float* r, float* g, float* b) {  // tonemapping(Vec8f&...), Color.hpp:66-73
	float x = aces_curve(*r * 0.59719f + *g * 0.35458f + *b * 0.04823f);
	float y = aces_curve(*r * 0.07600f + *g * 0.90834f + *b * 0.01566f);
	float z = aces_curve(*r * 0.02840f + *g * 0.13383f + *b * 0.83777f);
	*r = lane_min(1.0f, lane_max(0.0f, x * 1.604750f + y * -0.53108f + z * -0.07367f));
	*g = lane_min(1.0f, lane_max(0.0f, x * -0.10208f + y * 1.10813f + z * -0.00605f));
	*b = lane_min(1.0f, lane_max(0.0f, x * -0.00327f + y * -0.07276f + z * 1.07602f));
}

}  // namespace b2r
