// b2r_device.cuh — sm_100a kernels of the wavefront path tracer.
//
// Data layout in HBM (DESIGN.md "Layout"):
//   path queue (x2, ping-pong), SoA planes over the queue slot i:
//       A[i] = {o.x, o.y, o.z, d.x}   B[i] = {d.y, d.z, pdf, as_float(pid)}   T[c*cap + i] = throughput channel c
//     = 44 B per path (RayStream<>::Buffer, DataStreams.hpp:75-88, minus radiance). pid = slot << 26 | t with t the
//     pixel's tile-order index (tile*256 + ID) and slot the sample-in-flight index inside the batch.
//     BVH pipeline: + N[i] = the wide node the path's closest-hit walk starts at (4 B, written by k_shade).
//   radiance RAD[(slot*3 + c)*npix + t]: a path's running radiance lives at its pixel (one path per pixel per sample)
//     and is touched only when a contribution arrives (unoccluded light sample, emissive hit, sky).
//   hit queue H[i] = {tfar, as_float(prim)} and shadow queue SA/SB/SL (ray, light-sample radiance): BVH pipeline only.
//   buckets ACC[(k*3 + c)*npix + t]: running sums per median-of-means bucket (AccumulationTile, Renderer.hpp:43-46).
// All kernels are persistent (grid = SM count x resident CTAs, looping over a device-side count), so a whole batch —
// max_bounces rounds — is enqueued, or replayed as one CUDA graph, without host synchronisation.
#pragma once
#include <cuda_runtime.h>
#include "b2r_shade.h"

namespace b2r {

constexpr int kBruteTile = 256;        // spheres staged per shared-memory tile in the brute-force kernels
constexpr int kBlock = 256;            // threads per CTA, shading kernels
constexpr int kTravBlock = 128;        // threads per CTA, traversal kernels

// ---------------------------------------------------------------------------------------------- device-only helpers
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ void stat_add(unsigned long long* stats, int which, uint32_t v) {
	// one atomic per warp: REDUX.SUM over the lanes, lane 0 publishes
	const uint32_t s = __reduce_add_sync(0xffffffffu, v);
	if (lane_id() == 0 && s) atomicAdd(stats + which, static_cast<unsigned long long>(s));
}

// Shared-memory reads through a 32-bit shared-window address. nvcc for sm_100a re-derives the window base of a __shared__ array
// (S2UR SR_CgaCtaId + UMOV + ULEA) next to its uses, loops included; an address taken once and kept in a (uniform) register does not.
__device__ __forceinline__ uint32_t smem_addr(const void* p) {
	uint32_t a; asm volatile("mov.u32 %0, %1;" : "=r"(a) : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(p))));  // opaque: computed once, not rematerialised
	return a;
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
	float4 v; asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
	return v;
}
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ PathState load_path(const QueueDev& q, int side, uint32_t i) {
	const float4 a = q.A[side][i], b = q.B[side][i];
	PathState s; s.ox = a.x; s.oy = a.y; s.oz = a.z; s.dx = a.w; s.dy = b.x; s.dz = b.y; s.pdf = b.z; s.pid = __float_as_uint(b.w);
	const float* t = q.T[side];
	s.tr = t[i]; s.tg = t[q.cap + i]; s.tb = t[2u * q.cap + i];
	return s;
}

__device__ __forceinline__ void store_path(const QueueDev& q, int side, uint32_t i, const PathState& s) {
	q.A[side][i] = make_float4(s.ox, s.oy, s.oz, s.dx);
	q.B[side][i] = make_float4(s.dy, s.dz, s.pdf, __uint_as_float(s.pid));
	float* t = q.T[side];
	t[i] = s.tr; t[q.cap + i] = s.tg; t[2u * q.cap + i] = s.tb;
}

// ---------------------------------------------------------------------------------------------- brute-force pipeline
// One fused kernel per bounce (BVH.hpp:311-318 as shipped, USEBVH false): every ray is tested against every sphere, then the
// hits are shaded: closest-hit shader -> light sample + inline any-hit -> emissive -> BRDF sample / roulette -> append.
// Two things keep the SIMT lanes busy:
//   * the scene (spheres, materials, lights) is staged in shared memory and read as warp-uniform broadcasts;
//   * between intersection and shading the CTA compacts its hits through shared memory (index, distance, sphere), so the
//     long shading code runs on dense warps while warps left without hits skip it — misses cost one intersection loop.
#ifndef B2R_BRUTE_MIN_BLOCKS
#define B2R_BRUTE_MIN_BLOCKS 7      // resident CTAs per SM the register allocation is bounded for
#endif
#ifndef B2R_SHADE_MIN_BLOCKS
#define B2R_SHADE_MIN_BLOCKS 7      // k_shade: resident CTAs per SM the register allocation is bounded for
#endif
constexpr int kBruteBlock = 128;       // threads per CTA
constexpr int kBruteWarps = kBruteBlock / 32;
constexpr int kSmemTable = 64;         // materials / lights kept in shared memory when they fit

// rank of each flagged thread inside the CTA and the CTA total; one barrier. `s_cnt` must not be reused before another barrier.
__device__ __forceinline__ uint32_t block_rank(bool flag, uint32_t* s_cnt, uint32_t* total) {
	const uint32_t ballot = __ballot_sync(0xffffffffu, flag);
	const uint32_t warp = threadIdx.x >> 5;
	if (lane_id() == 0) s_cnt[warp] = __popc(ballot);
	__syncthreads();
	uint32_t off = 0, tot = 0;
#pragma unroll
	for (uint32_t w = 0; w < kBruteWarps; w++) { const uint32_t c = s_cnt[w]; off += (w < warp) ? c : 0u; tot += c; }
	*total = tot;
	return off + __popc(ballot & ((1u << lane_id()) - 1u));
}

// two flags ranked behind ONE barrier (the shading phase ranks its shadow rays and its surviving paths together)
__device__ __forceinline__ void block_rank2(bool fa, bool fb, uint32_t* s_a, uint32_t* s_b, uint32_t* rank_a, uint32_t* total_a, uint32_t* rank_b, uint32_t* total_b) {
	const uint32_t ba = __ballot_sync(0xffffffffu, fa), bb = __ballot_sync(0xffffffffu, fb);
	const uint32_t warp = threadIdx.x >> 5, below = (1u << lane_id()) - 1u;
	if (lane_id() == 0) { s_a[warp] = __popc(ba); s_b[warp] = __popc(bb); }
	__syncthreads();
	uint32_t oa = 0, ta = 0, ob = 0, tb = 0;
#pragma unroll
	for (uint32_t w = 0; w < kBruteWarps; w++) { const uint32_t ca = s_a[w], cb = s_b[w]; oa += (w < warp) ? ca : 0u; ta += ca; ob += (w < warp) ? cb : 0u; tb += cb; }
	*total_a = ta; *total_b = tb;
	*rank_a = oa + __popc(ba & below); *rank_b = ob + __popc(bb & below);
}

// The late bounces of the brute-force pipeline are thin (C2: bounces >= 5 carry 3 % of the instructions of a batch but 10 % of its time, at
// 20-45 % issue utilisation: each launch stages the scene, fills and drains its shared-memory queues for a handful of rays per CTA). Once
// fewer than frame.finish_below paths enter a bounce (first checked at frame.finish_first), k_brute_finish traces those paths to their end in
// ONE launch and the per-bounce kernels of the remaining bounces return at once: the path counts only fall, so "paths[bounce] <
// finish_below" says the same thing in every kernel (an untouched count of a later bounce reads 0).
__device__ __forceinline__ bool finished_elsewhere(const Params& p, uint32_t bounce, uint32_t n_in) {
	return p.frame.finish_below != 0u && bounce >= p.frame.finish_first && bounce + 1u < p.frame.max_bounces && n_in < p.frame.finish_below;  // (the last bounce is never handed over: nothing is left to finish)
}

// EXACT (B2R_FLAG_REFERENCE_EXACT): rays that sit in the last `active % 8` slots of their tile's stream take the reference's
// scalar-tail sphere formula (BVH.hpp:270-286) instead of the AVX2+FMA one (:250-268), and survivors leave (material, slot) behind
// for k_stream_rank, which computes the slots of the next bounce (the reference's stable counting sort by material).
// LENS (bounce 0 with a thin lens): every camera ray has its own origin, so there is no shared-origin sphere precompute (s_pre); phase 1
// runs sphere_hit_closest per ray, and phase 2 regenerates a hit's camera ray from its path id instead of queueing its origin.
// DIELECTRIC (B2R_FLAG_DIELECTRIC): the shading routines' smooth-dielectric path (b2r_shade.h dielectric_scatter); the same axis in k_brute_finish
// and k_shade.
template <bool FIRST, bool COUNT, bool EXACT, bool GGX = false, bool LENS = false, bool DIELECTRIC = false>
__global__ void __launch_bounds__(kBruteBlock, B2R_BRUTE_MIN_BLOCKS) k_bounce_brute(const Params p, const uint32_t bounce) {
	constexpr int kQ = 2 * kBruteBlock;  // hit queue: up to kBruteBlock-1 waiting + kBruteBlock new
	__shared__ float4 s_prim[kBruteTile];
	constexpr bool PRE = FIRST && !LENS;
	__shared__ float4 s_pre[PRE ? kBruteTile : 1];  // bounce 0: {c - o, r^2 - |c - o|^2} per sphere for the shared camera origin
	__shared__ int32_t s_prim_mat[kBruteTile];
	__shared__ float4 s_table[4][kSmemTable];  // mat_albedo, mat_emission, light_sphere, light_emit
	__shared__ uint32_t s_hit_i[kQ]; __shared__ float s_hit_t[kQ]; __shared__ int32_t s_hit_prim[kQ];
	__shared__ float s_hit_d[PRE ? 3 : 1][PRE ? kQ : 1];
	__shared__ float s_shadow[11][kQ];         // shadow-ray queue: o.xyz, d.xyz, tfar, L.rgb, pid
	__shared__ uint32_t s_cnt_a[kBruteWarps], s_cnt_b[kBruteWarps], s_cnt_c[kBruteWarps], s_base;
	SceneDev sc = p.scene;
	const uint32_t n_in = FIRST ? p.batch->n_slots * p.frame.npix : p.cnt.paths[bounce];
	const int side = bounce & 1;
	const uint32_t n_tiles = (sc.n_prims + kBruteTile - 1) / kBruteTile;
	const bool mis = !(p.frame.flags & B2R_FLAG_NO_MIS);
	const bool last = bounce + 1 >= p.frame.max_bounces;
	uint32_t c_shadow = 0, c_hits = 0, c_term = 0, c_drop = 0, c_events = 0, c_sphere = 0;
	if (blockIdx.x * kBruteBlock >= n_in) return;  // thin late bounces: CTAs without a first chunk leave before staging anything
	if (!FIRST && !EXACT && finished_elsewhere(p, bounce, n_in)) return;  // k_brute_finish has taken the rest of the batch

	// stage the scene tables once per CTA (persistent: amortised over the whole launch)
	if (n_tiles == 1) {
		for (uint32_t j = threadIdx.x; j < sc.n_prims; j += blockDim.x) {
			const float4 sp = sc.prims[j]; s_prim[j] = sp; s_prim_mat[j] = sc.prim_mat[j];
			if (PRE) { const SpherePre q = sphere_prepare(sp.x, sp.y, sp.z, sp.w, p.batch->cam.px, p.batch->cam.py, p.batch->cam.pz); s_pre[j] = make_float4(q.tx, q.ty, q.tz, q.disc0); }
		}
		sc.prim_mat = s_prim_mat; sc.prims = s_prim;
	}
	if (sc.n_mat <= kSmemTable) {
		for (uint32_t j = threadIdx.x; j < sc.n_mat; j += blockDim.x) { s_table[0][j] = sc.mat_albedo[j]; s_table[1][j] = sc.mat_emission[j]; }
		sc.mat_albedo = s_table[0]; sc.mat_emission = s_table[1];
	}
	if (sc.n_lights <= kSmemTable) {
		for (uint32_t j = threadIdx.x; j < sc.n_lights; j += blockDim.x) { s_table[2][j] = sc.light_sphere[j]; s_table[3][j] = sc.light_emit[j]; }
		sc.light_sphere = s_table[2]; sc.light_emit = s_table[3];
	}
	__syncthreads();

	const uint32_t a_prim = smem_addr(s_prim), a_pre = smem_addr(s_pre);
	uint32_t queued = 0, s_queued = 0;         // hits / shadow rays waiting in shared memory (CTA-uniform)
	uint32_t base = blockIdx.x * kBruteBlock;
	for (;;) {
		const bool more = base < n_in;         // CTA-uniform
		if (more) {
			// ---------------- phase 1: one ray per thread, closest hit over every sphere (ties -> lowest BVH-order index, strict <, Q6)
			const uint32_t i = base + threadIdx.x;
			const bool live = i < n_in;
			float ox = 0, oy = 0, oz = 0, dx = 0, dy = 0, dz = 0; uint32_t pid0 = 0; bool tail = false;
			if (live) {
				if (FIRST) {
					const uint32_t sl0 = div_by(i, p.frame.npix, p.frame.npix_magic);
					const PathState s0 = primary_path<LENS>(p.frame, p.batch->cam, p.batch->acc[sl0], sl0, i - sl0 * p.frame.npix, p.batch->lens);
					ox = s0.ox; oy = s0.oy; oz = s0.oz; dx = s0.dx; dy = s0.dy; dz = s0.dz;
					pid0 = s0.pid; rad_zero(p.rad, p.frame.npix, s0.pid);  // a path's radiance starts at 0 here (coalesced stores); contributions are added after a CTA barrier
				} else {
					const float4 a = p.q.A[side][i], b = p.q.B[side][i];
					ox = a.x; oy = a.y; oz = a.z; dx = a.w; dy = b.x; dz = b.y;
					if (EXACT) {  // stream = (sample in flight, tile); in the scalar tail when slot >= active & ~7
						const uint32_t pid_i = __float_as_uint(b.w), stream = (pid_i >> 26) * (p.frame.npix >> 8) + ((pid_i & kPixMask) >> 8);
						tail = static_cast<uint32_t>(p.ex.slot[side][i]) >= (static_cast<uint32_t>(p.ex.act[side][stream]) & ~7u);
					}
				}
			}
			float best = FLT_MAX; int32_t prim = -1;
			for (uint32_t tile = 0; tile < n_tiles; tile++) {
				const uint32_t first = tile * kBruteTile, cnt = min(static_cast<uint32_t>(kBruteTile), sc.n_prims - first);
				if (n_tiles > 1) {
					__syncthreads();
					for (uint32_t j = threadIdx.x; j < cnt; j += blockDim.x) {
						const float4 sp = p.scene.prims[first + j]; s_prim[j] = sp;
						if (PRE) { const SpherePre q = sphere_prepare(sp.x, sp.y, sp.z, sp.w, p.batch->cam.px, p.batch->cam.py, p.batch->cam.pz); s_pre[j] = make_float4(q.tx, q.ty, q.tz, q.disc0); }
					}
					__syncthreads();
				}
				if (EXACT && live && tail) {
					for (uint32_t j = 0; j < cnt; j++) { const float4 sp = lds_f4(a_prim + j * 16u); sphere_closest_scalar_update(sp.x, sp.y, sp.z, sp.w, static_cast<int32_t>(first + j), ox, oy, oz, dx, dy, dz, &best, &prim); }
					if (COUNT) c_sphere += cnt;
				} else if (live) {
				#pragma unroll 3
					for (uint32_t j = 0; j < cnt; j++) {
						float d; bool h;
						if (PRE) { const float4 q = lds_f4(a_pre + j * 16u); h = sphere_hit_prepared(SpherePre{q.x, q.y, q.z, q.w}, dx, dy, dz, &d); }
						else { const float4 sp = lds_f4(a_prim + j * 16u); h = sphere_hit_closest(sp.x, sp.y, sp.z, sp.w, ox, oy, oz, dx, dy, dz, &d); }
						if (h && d < best) { best = d; prim = static_cast<int32_t>(first + j); }
					}
					if (COUNT) c_sphere += cnt;
				}
			}
			const bool is_hit = live && prim >= 0;
			if (live && !is_hit) {  // miss shader (Renderer.hpp:408-420): the path ends, its radiance stays at the pixel
				c_term++;
				if (sc.has_ambient) {
					const uint32_t slm = FIRST ? div_by(i, p.frame.npix, p.frame.npix_magic) : 0u;
					const PathState sm = FIRST ? primary_path<LENS>(p.frame, p.batch->cam, p.batch->acc[slm], slm, i - slm * p.frame.npix, p.batch->lens) : load_path(p.q, side, i);
					rad_add(p.rad, p.frame.npix, sm.pid, shade_sky(sc, sm), f3{0.0f, 0.0f, 0.0f}, true, false); c_events++;
				}
			}
			// ---------------- the CTA's hits join the shared-memory queue
			uint32_t n_hits;
			const uint32_t slot = queued + block_rank(is_hit, s_cnt_a, &n_hits);
			if (is_hit) {
				s_hit_i[slot] = FIRST ? pid0 : i; s_hit_t[slot] = best; s_hit_prim[slot] = prim;  // bounce 0 queues the path id itself (no queue record to index)
				if (PRE) { s_hit_d[0][slot] = dx; s_hit_d[PRE ? 1 : 0][slot] = dy; s_hit_d[PRE ? 2 : 0][slot] = dz; }
			}
			queued += n_hits;
			base += gridDim.x * kBruteBlock;
			__syncthreads();
		}
		// ---------------- phase 2: shade queued hits — only full CTAs of them (every warp dense), or the rest once rays run out
		if (queued >= static_cast<uint32_t>(kBruteBlock) || (!more && queued > 0)) {
			const uint32_t take = min(queued, static_cast<uint32_t>(kBruteBlock));
			const uint32_t qi = queued - take + threadIdx.x;
			const bool shade = threadIdx.x < take;
			queued -= take;
			bool keep = false, want_shadow = false;
			PathState s; ShadowRay sr; uint32_t pid = 0; uint32_t ex_slot = 0, ex_mat = 0;
			if (shade) {
				const uint32_t hi = s_hit_i[qi]; const float depth = s_hit_t[qi]; const int32_t hprim = s_hit_prim[qi];
				if (EXACT) ex_slot = FIRST ? (hi & 255u) : static_cast<uint32_t>(p.ex.slot[side][hi]);  // bounce 0: hi is the path id, slot = pixel ID
				if (PRE) {
					s.ox = p.batch->cam.px; s.oy = p.batch->cam.py; s.oz = p.batch->cam.pz;
					s.dx = s_hit_d[0][PRE ? qi : 0]; s.dy = s_hit_d[PRE ? 1 : 0][PRE ? qi : 0]; s.dz = s_hit_d[PRE ? 2 : 0][PRE ? qi : 0];
					s.tr = s.tg = s.tb = 1.0f; s.pdf = 0.0f; s.pid = hi;
				} else if (FIRST) s = primary_path<LENS>(p.frame, p.batch->cam, p.batch->acc[hi >> 26], hi >> 26, hi & kPixMask, p.batch->lens);  // the same bits phase 1 traced
				else s = load_path(p.q, side, hi);
				pid = s.pid;
				const uint32_t acc = p.batch->acc[s.pid >> 26], seed = pixel_seed(s.pid & kPixMask, p.frame.max_bounces);
				const Surface sf = shade_surface<GGX, DIELECTRIC>(sc, s, depth, hprim, p.mat_diel);
				if (EXACT) ex_mat = static_cast<uint32_t>(sf.mat);
				c_hits++;
				if (last) { rad_zero(p.rad, p.frame.npix, s.pid); c_drop++; }  // survivors of the last bounce lose their radiance (Q11)
				else {
					if (mis) want_shadow = shade_light_sample<GGX, DIELECTRIC>(sc, sf, s, hprim, acc, seed, bounce, &sr);
					if (sf.emissive) {
						// light sample first, then emission (Renderer.hpp:304-353). The shadow test of an emissive hit (rare) is done
						// right here so that order holds; every other shadow ray goes to the queue and is tested by dense warps.
						const f3 e_add = shade_emission<DIELECTRIC>(sc, sf, s, depth, bounce, mis);
						if (want_shadow) {
							c_shadow++;
							bool occluded = false;
							for (uint32_t j = 0; j < sc.n_prims && !occluded; j++) {
								const float4 sp = sc.prims[j];  // shared-memory copy when the scene fits one tile, global otherwise
								occluded = sphere_hit_any(sp.x, sp.y, sp.z, sp.w, sr.o.x, sr.o.y, sr.o.z, sr.d.x, sr.d.y, sr.d.z, sr.tfar);
							}
							if (COUNT) c_sphere += sc.n_prims;
							rad_add(p.rad, p.frame.npix, s.pid, sr.L, e_add, !occluded, true);
							want_shadow = false;
						} else rad_add(p.rad, p.frame.npix, s.pid, e_add, f3{0.0f, 0.0f, 0.0f}, true, false);
						c_events++;
					}
					keep = shade_continue<GGX, DIELECTRIC>(sf, &s, acc, seed, bounce);
					if (!keep) c_term++;  // roulette: path ends here, radiance stays at the pixel (Renderer.hpp:379-381,424-430)
				}
			}
			// shadow rays -> shared-memory queue; survivors -> next path queue (one atomic per CTA)
			uint32_t n_shadow, n_keep, srank, rank;
			block_rank2(want_shadow, keep, s_cnt_c, s_cnt_b, &srank, &n_shadow, &rank, &n_keep);  // barrier: hit-queue reads above precede the next phase 1
			const uint32_t sslot = s_queued + srank;
			if (want_shadow) {
				s_shadow[0][sslot] = sr.o.x; s_shadow[1][sslot] = sr.o.y; s_shadow[2][sslot] = sr.o.z;
				s_shadow[3][sslot] = sr.d.x; s_shadow[4][sslot] = sr.d.y; s_shadow[5][sslot] = sr.d.z; s_shadow[6][sslot] = sr.tfar;
				s_shadow[7][sslot] = sr.L.x; s_shadow[8][sslot] = sr.L.y; s_shadow[9][sslot] = sr.L.z; s_shadow[10][sslot] = __uint_as_float(pid);
			}
			s_queued += n_shadow;
			if (threadIdx.x == 0) s_base = n_keep ? atomicAdd(p.cnt.paths + bounce + 1, n_keep) : 0u;
			__syncthreads();
			if (keep) {
				store_path(p.q, side ^ 1, s_base + rank, s);
				if (EXACT) {  // (stream, slot) -> material and next-queue index, for k_stream_rank
					const uint32_t e = (pid >> 26) * p.frame.npix + ((pid & kPixMask) & ~255u) + ex_slot;
					p.ex.key[e] = static_cast<uint8_t>(ex_mat + 1u); p.ex.next_idx[e] = s_base + rank;
				}
			}
		}
		// ---------------- phase 3: any-hit test of queued shadow rays (BVH.hpp:290-305), again a full CTA at a time
		const bool drained = !more && queued == 0;
		if (s_queued >= static_cast<uint32_t>(kBruteBlock) || (drained && s_queued > 0)) {
			const uint32_t take = min(s_queued, static_cast<uint32_t>(kBruteBlock));
			const uint32_t qi = s_queued - take + threadIdx.x;
			const bool test = threadIdx.x < take;
			s_queued -= take;
			float sox = 0, soy = 0, soz = 0, sdx = 0, sdy = 0, sdz = 0, stfar = 0; f3 L{0.0f, 0.0f, 0.0f}; uint32_t spid = 0;
			if (test) {
				sox = s_shadow[0][qi]; soy = s_shadow[1][qi]; soz = s_shadow[2][qi]; sdx = s_shadow[3][qi]; sdy = s_shadow[4][qi]; sdz = s_shadow[5][qi];
				stfar = s_shadow[6][qi]; L = f3{s_shadow[7][qi], s_shadow[8][qi], s_shadow[9][qi]}; spid = __float_as_uint(s_shadow[10][qi]);
				c_shadow++;
			}
			bool occluded = !test;
			if (n_tiles == 1) {
				if (COUNT && test) c_sphere += sc.n_prims;
				for (uint32_t j0 = 0; j0 < sc.n_prims; j0 += 3u) {  // three spheres per early-out vote
#pragma unroll
					for (uint32_t u = 0; u < 3u; u++) {
						if (j0 + u < sc.n_prims) {
							const float4 sp = lds_f4(a_prim + (j0 + u) * 16u);
							if (!occluded && sphere_hit_any(sp.x, sp.y, sp.z, sp.w, sox, soy, soz, sdx, sdy, sdz, stfar)) occluded = true;
						}
					}
					if (__all_sync(0xffffffffu, occluded)) break;
				}
			} else {
				for (uint32_t tile = 0; tile < n_tiles; tile++) {
					const uint32_t first = tile * kBruteTile, cnt = min(static_cast<uint32_t>(kBruteTile), sc.n_prims - first);
					__syncthreads();
					for (uint32_t j = threadIdx.x; j < cnt; j += blockDim.x) s_prim[j] = p.scene.prims[first + j];
					__syncthreads();
					if (!occluded) {
						if (COUNT) c_sphere += cnt;
						for (uint32_t j = 0; j < cnt && !occluded; j++) {
							const float4 sp = s_prim[j];
							occluded = sphere_hit_any(sp.x, sp.y, sp.z, sp.w, sox, soy, soz, sdx, sdy, sdz, stfar);
						}
					}
				}
			}
			if (test && !occluded) { rad_add(p.rad, p.frame.npix, spid, L, f3{0.0f, 0.0f, 0.0f}, true, false); c_events++; }
			__syncthreads();  // shadow-queue reads above precede the next phase 2 writes
		}
		if (drained && s_queued == 0) break;
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(p.cnt.stats + ST_EXT, static_cast<unsigned long long>(n_in));
	stat_add(p.cnt.stats, ST_SHADOW, c_shadow); stat_add(p.cnt.stats, ST_HITS, c_hits); stat_add(p.cnt.stats, ST_TERM, c_term);
	stat_add(p.cnt.stats, ST_DROPPED, c_drop); stat_add(p.cnt.stats, ST_EVENTS, c_events);
	if (COUNT) stat_add(p.cnt.stats, ST_SPHERE, c_sphere);
}


// The rest of every path that enters bounce `bounce0` of the brute-force pipeline, in one launch (see finished_elsewhere). One path per
// lane; both sphere loops are warp-uniform (every lane walks all the spheres of the shared-memory copy), so the only divergence is paths
// ending, and a lane whose path has ended picks up the next waiting path. Same routines, same RNG streams (a function of sample, pixel and
// bounce), same order of a path's radiance additions (light sample, then emission) as k_bounce_brute: every path ends with the same bits.
template <bool COUNT, bool GGX = false, bool DIELECTRIC = false>
__global__ void __launch_bounds__(kBruteBlock, B2R_BRUTE_MIN_BLOCKS) k_brute_finish(const Params p, const uint32_t bounce0) {
	__shared__ float4 s_prim[kBruteTile];
	__shared__ int32_t s_prim_mat[kBruteTile];
	__shared__ float4 s_table[4][kSmemTable];
	SceneDev sc = p.scene;
	const uint32_t n_in = p.cnt.paths[bounce0];
	if (n_in == 0u || !finished_elsewhere(p, bounce0, n_in)) return;
	if (bounce0 > p.frame.finish_first && p.cnt.paths[bounce0 - 1u] < p.frame.finish_below) return;  // an earlier launch of this kernel took them
	if (blockIdx.x * kBruteBlock >= n_in) return;
	const int side = bounce0 & 1;
	const bool mis = !(p.frame.flags & B2R_FLAG_NO_MIS);
	const uint32_t mb = p.frame.max_bounces, n_prims = sc.n_prims;
	for (uint32_t j = threadIdx.x; j < n_prims; j += blockDim.x) { s_prim[j] = sc.prims[j]; s_prim_mat[j] = sc.prim_mat[j]; }  // (launched only when the scene fits one tile)
	sc.prim_mat = s_prim_mat; sc.prims = s_prim;
	if (sc.n_mat <= kSmemTable) {
		for (uint32_t j = threadIdx.x; j < sc.n_mat; j += blockDim.x) { s_table[0][j] = sc.mat_albedo[j]; s_table[1][j] = sc.mat_emission[j]; }
		sc.mat_albedo = s_table[0]; sc.mat_emission = s_table[1];
	}
	if (sc.n_lights <= kSmemTable) {
		for (uint32_t j = threadIdx.x; j < sc.n_lights; j += blockDim.x) { s_table[2][j] = sc.light_sphere[j]; s_table[3][j] = sc.light_emit[j]; }
		sc.light_sphere = s_table[2]; sc.light_emit = s_table[3];
	}
	__syncthreads();
	const uint32_t a_prim = smem_addr(s_prim);
	uint32_t c_ext = 0, c_shadow = 0, c_hits = 0, c_term = 0, c_drop = 0, c_events = 0, c_sphere = 0;
	uint32_t next = 0, end = 0; bool dry = false;  // warp-uniform: 32 paths per claim
	PathState s; uint32_t bounce = 0; bool alive = false;
	for (;;) {
		// lanes without a path take the next waiting ones
		const uint32_t idle = __ballot_sync(0xffffffffu, !alive);
		if (idle && !dry) {
			uint32_t want = __popc(idle), given = 0, mine = 0xffffffffu;
			while (want > given && !dry) {
				if (next >= end) {
					uint32_t b = 0;
					if (lane_id() == 0) b = atomicAdd(p.cnt.work_a + bounce0, 32u);
					b = __shfl_sync(0xffffffffu, b, 0);
					if (b >= n_in) { dry = true; break; }
					next = b; end = min(b + 32u, n_in);
				}
				const uint32_t n = min(want - given, end - next), rank = __popc(idle & ((1u << lane_id()) - 1u));
				if (!alive && rank >= given && rank < given + n) mine = next + (rank - given);
				next += n; given += n;
			}
			if (mine != 0xffffffffu) { s = load_path(p.q, side, mine); bounce = bounce0; alive = true; }
		}
		if (!__any_sync(0xffffffffu, alive)) break;
		// closest hit over every sphere (ties -> lowest BVH-order index, strict <, Q6)
		float best = FLT_MAX; int32_t prim = -1;
		if (alive) {
			c_ext++;
			for (uint32_t j = 0; j < n_prims; j++) {
				const float4 sp = lds_f4(a_prim + j * 16u); float d;
				if (sphere_hit_closest(sp.x, sp.y, sp.z, sp.w, s.ox, s.oy, s.oz, s.dx, s.dy, s.dz, &d) && d < best) { best = d; prim = static_cast<int32_t>(j); }
			}
			if (COUNT) c_sphere += n_prims;
		}
		bool want_shadow = false, has_emit = false, keep = false; ShadowRay sr{}; f3 emit{0.0f, 0.0f, 0.0f}; const uint32_t pid = s.pid;
		if (alive) {
			if (prim < 0) {  // miss shader (Renderer.hpp:408-420)
				c_term++;
				if (sc.has_ambient) { rad_add(p.rad, p.frame.npix, pid, shade_sky(sc, s), f3{0.0f, 0.0f, 0.0f}, true, false); c_events++; }
			} else {
				const uint32_t acc = p.batch->acc[pid >> 26], seed = pixel_seed(pid & kPixMask, mb);
				const Surface sf = shade_surface<GGX, DIELECTRIC>(sc, s, best, prim, p.mat_diel);
				c_hits++;
				if (bounce + 1u >= mb) { rad_zero(p.rad, p.frame.npix, pid); c_drop++; }  // Q11
				else {
					if (mis) want_shadow = shade_light_sample<GGX, DIELECTRIC>(sc, sf, s, prim, acc, seed, bounce, &sr);
					if (sf.emissive) { emit = shade_emission<DIELECTRIC>(sc, sf, s, best, bounce, mis); has_emit = true; }
					keep = shade_continue<GGX, DIELECTRIC>(sf, &s, acc, seed, bounce);
					if (!keep) c_term++;
				}
			}
		}
		// any-hit test of this bounce's shadow ray (BVH.hpp:290-305), three spheres per early-out vote
		bool occluded = !want_shadow;
		if (__any_sync(0xffffffffu, want_shadow)) {
			if (want_shadow) { c_shadow++; if (COUNT) c_sphere += n_prims; }
			for (uint32_t j0 = 0; j0 < n_prims; j0 += 3u) {
#pragma unroll
				for (uint32_t u = 0; u < 3u; u++) {
					if (j0 + u < n_prims) {
						const float4 sp = lds_f4(a_prim + (j0 + u) * 16u);
						if (!occluded && sphere_hit_any(sp.x, sp.y, sp.z, sp.w, sr.o.x, sr.o.y, sr.o.z, sr.d.x, sr.d.y, sr.d.z, sr.tfar)) occluded = true;
					}
				}
				if (__all_sync(0xffffffffu, occluded)) break;
			}
		}
		const bool lit = want_shadow && !occluded;
		// light sample first, then emission (Renderer.hpp:304-353); one radiance event per emissive hit, as k_bounce_brute counts them
		if (has_emit) { rad_add(p.rad, p.frame.npix, pid, sr.L, emit, lit, true); c_events++; }
		else if (lit) { rad_add(p.rad, p.frame.npix, pid, sr.L, f3{0.0f, 0.0f, 0.0f}, true, false); c_events++; }
		alive = keep; bounce++;
	}
	stat_add(p.cnt.stats, ST_EXT, c_ext); stat_add(p.cnt.stats, ST_SHADOW, c_shadow); stat_add(p.cnt.stats, ST_HITS, c_hits); stat_add(p.cnt.stats, ST_TERM, c_term);
	stat_add(p.cnt.stats, ST_DROPPED, c_drop); stat_add(p.cnt.stats, ST_EVENTS, c_events);
	if (COUNT) stat_add(p.cnt.stats, ST_SPHERE, c_sphere);
}

// B2R_FLAG_REFERENCE_EXACT, after bounce `bounce`: the reference compacts a tile's survivors in the order of its stable counting
// sort by material (sort_rayID, DataStreams.hpp:236-253, called at Renderer.hpp:235-243; the BRDF loop appends in that order,
// :359-404): rank = (survivors with a smaller material) + (same material, smaller slot). One WARP per stream, warp-synchronous:
// eight rounds of 32 consecutive slots; in a round the lanes with the same material find each other with MATCH.ANY and take their
// place after the running count of that material; a 64-bin scan then turns the per-material totals into bases.
__global__ void __launch_bounds__(256) k_stream_rank(const Params p, const uint32_t bounce) {
	__shared__ uint16_t s_run[8][64];
	const int side = bounce & 1;
	const uint32_t n_streams = p.batch->n_slots * (p.frame.npix >> 8), warp = threadIdx.x >> 5, lane = lane_id(), below = (1u << lane) - 1u;
	uint16_t* run = s_run[warp];
	// a warp takes 32 consecutive streams at a time: one coalesced look at their active counts, then only the non-empty ones are ranked
	for (uint32_t group = (blockIdx.x * 8u + warp) * 32u; group < n_streams; group += gridDim.x * 8u * 32u) {
		const uint32_t mine = group + lane;
		const bool has_rays = mine < n_streams && (bounce == 0u || p.ex.act[side][mine] != 0u);
		if (mine < n_streams && !has_rays) p.ex.act[side ^ 1][mine] = 0;
		uint32_t todo = __ballot_sync(0xffffffffu, has_rays);
		while (todo) {
			const uint32_t stream = group + static_cast<uint32_t>(__ffs(static_cast<int>(todo)) - 1);
			todo &= todo - 1u;
			const uint32_t e0 = stream * 256u + lane;
			uint32_t key[8], any = 0u;
#pragma unroll
			for (uint32_t r = 0; r < 8u; r++) { key[r] = p.ex.key[e0 + 32u * r]; any |= key[r]; }
			if (!__any_sync(0xffffffffu, any != 0u)) { if (lane == 0u) p.ex.act[side ^ 1][stream] = 0; continue; }
			run[lane] = 0; run[lane + 32u] = 0;
			__syncwarp();
			uint32_t within[8];
#pragma unroll
			for (uint32_t r = 0; r < 8u; r++) {
				const bool alive = key[r] != 0u;
				within[r] = 0u;
				if (!__any_sync(0xffffffffu, alive)) continue;  // nobody left in these 32 slots (late bounces: most rounds)
				const uint32_t m = alive ? key[r] - 1u : 0xffffu;  // the dead lanes match each other: harmless
				const uint32_t peers = __match_any_sync(0xffffffffu, m), rk = __popc(peers & below);
				if (alive) within[r] = run[m] + rk;
				__syncwarp();
				if (alive && rk == 0u) run[m] = static_cast<uint16_t>(run[m] + __popc(peers));
				if (alive) p.ex.key[e0 + 32u * r] = 0;  // left clean for the next bounce
				__syncwarp();
			}
			const uint32_t c0 = run[2u * lane], c1 = run[2u * lane + 1u];
			uint32_t incl = c0 + c1;
#pragma unroll
			for (uint32_t d = 1; d < 32u; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
			const uint32_t total = __shfl_sync(0xffffffffu, incl, 31), excl = incl - (c0 + c1);
			__syncwarp();
			run[2u * lane] = static_cast<uint16_t>(excl); run[2u * lane + 1u] = static_cast<uint16_t>(excl + c0);
			__syncwarp();
#pragma unroll
			for (uint32_t r = 0; r < 8u; r++) if (key[r] != 0u) p.ex.slot[side ^ 1][p.ex.next_idx[e0 + 32u * r]] = static_cast<uint8_t>(run[key[r] - 1u] + within[r]);
			if (lane == 0u) p.ex.act[side ^ 1][stream] = static_cast<uint16_t>(total);
			__syncwarp();
		}
	}
}

// camera rays of a batch -> queue side 0 (Renderer.hpp:97-127)
template <bool LENS = false>
__global__ void __launch_bounds__(kBlock) k_generate(const Params p) {
	const uint32_t n = p.batch->n_slots * p.frame.npix;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
		{ const uint32_t sl = div_by(i, p.frame.npix, p.frame.npix_magic); const PathState s = primary_path<LENS>(p.frame, p.batch->cam, p.batch->acc[sl], sl, i - sl * p.frame.npix, p.batch->lens); store_path(p.q, 0, i, s); rad_zero(p.rad, p.frame.npix, s.pid); }
	if (blockIdx.x == 0 && threadIdx.x == 0) p.cnt.paths[0] = n;
}
// Work distribution of the traversal kernels: every warp owns a pool of ray indices claimed kTravChunk at a time from the
// bounce's cursor (one atomic per chunk); lanes whose ray has finished are refilled from the pool as soon as fewer than
// kRefillBelow lanes of the warp are still traversing, so a warp never idles behind its longest ray.
#ifndef B2R_REFILL_BELOW
#define B2R_REFILL_BELOW 24
#endif
constexpr uint32_t kTravChunk = 128, kRefillBelow = B2R_REFILL_BELOW;
struct WarpPool {
	uint32_t next = 0, end = 0; bool dry = false;  // warp-uniform
	// Guided chunks: a warp claims 128 rays while plenty are left and fewer (down to 32 = one ray per lane) as the queue runs out, about
	// half of an even share of what is left. The end of every launch — and the whole of a thin late-bounce launch — is then spread over
	// all resident warps instead of a few warps walking 128 rays each, four rounds in a row, while the rest of the GPU idles.
	__device__ __forceinline__ uint32_t chunk_for(const uint32_t* cursor, uint32_t n_in) const {
		const uint32_t at = *reinterpret_cast<const volatile uint32_t*>(cursor);
		const uint32_t left = n_in > at ? n_in - at : 0u, warps = gridDim.x * (blockDim.x >> 5);
		const uint32_t share = left / (2u * warps);
		return share >= kTravChunk ? kTravChunk : share <= 32u ? 32u : (share & ~31u);
	}
	// hands ray indices to the lanes flagged `idle`; returns the lane's index or 0xffffffff
	__device__ __forceinline__ uint32_t take(bool idle, uint32_t* cursor, uint32_t n_in) {
		const uint32_t mask = __ballot_sync(0xffffffffu, idle);
		uint32_t mine = 0xffffffffu;
		uint32_t want = __popc(mask), given = 0;
		while (want > given && !dry) {
			if (next >= end) {
				uint32_t b = 0, chunk = 0;
				if (lane_id() == 0) { chunk = chunk_for(cursor, n_in); b = atomicAdd(cursor, chunk); }
				b = __shfl_sync(0xffffffffu, b, 0); chunk = __shfl_sync(0xffffffffu, chunk, 0);
				if (b >= n_in) { dry = true; break; }
				next = b; end = min(b + chunk, n_in);
			}
			const uint32_t n = min(want - given, end - next);
			const uint32_t rank = __popc(mask & ((1u << lane_id()) - 1u));
			if (idle && rank >= given && rank < given + n) mine = next + (rank - given);
			next += n; given += n;
		}
		return mine;
	}
};
// Node staging: the lanes of a warp sit on 32 different 128-byte nodes. Read naively that is 8 x LDG.128 with 32 lines each
// (256 L1 wavefronts per step — the first version was bound by exactly that). Instead the warp copies the 32 nodes
// cooperatively, 8 lanes x 16 B per node so each copy instruction touches 4 lines, straight into shared memory (cp.async,
// no register staging); every lane then reads its own node back with LDS.128.
constexpr int kNodeRowF4 = 9;  // 128-byte node in a 144-byte row: the 16-byte pad makes the cooperative fill and the per-lane LDS.128 reads conflict-free
                               // with plain immediate offsets (an XOR swizzle did the same at two extra address instructions per read)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
	const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
	asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void warp_stage_nodes(const WideNode* __restrict__ wide, float4* s_rows /*[32][kNodeRowF4] of this warp*/, uint32_t my_node) {
	// lanes without a ray pass node 0 (the root, always cached), so the copies need no predicate
	const uint32_t lane = lane_id(), part = lane & 7u;
#pragma unroll
	for (uint32_t j = 0; j < 8; j++) {
		const uint32_t owner = 4u * j + (lane >> 3);
		const uint32_t nd = __shfl_sync(0xffffffffu, my_node, owner);
		cp_async16(s_rows + owner * kNodeRowF4 + part, reinterpret_cast<const float4*>(wide + nd) + part);
	}
	asm volatile("cp.async.wait_all;" ::: "memory");
	__syncwarp();
}
// Per-thread traversal stack of the persistent kernels: kSmemStack entries in shared memory, laid out [entry][thread] so a
// warp's accesses are conflict-free whatever the lanes' depths. The hot path never tests for overflow per access: once per node
// visit room() makes sure three more entries fit, and if they do not (rare: the host bounds the worst case, typical rays use a
// handful) the kEvict oldest entries move to a local-memory backing store and come back through refill() when the shared part
// has run empty — LIFO order is kept because the oldest entries are the last to be popped.
#ifndef B2R_SMEM_STACK
#define B2R_SMEM_STACK 16
#endif
constexpr int kSmemStack = B2R_SMEM_STACK, kEvict = 8;
static_assert(kSmemStack >= kEvict + 3 && kTraversalStack % kEvict == 0, "stack geometry");
constexpr uint32_t kStackStride = kTravBlock * 4u;  // bytes between consecutive entries of one thread
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v)); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
// the rare paths are real calls that see only the backing array, so the per-ray state stays in registers
__device__ __noinline__ void stack_evict(uint32_t base, uint32_t top, uint32_t* backing) {
	for (int j = 0; j < kEvict; j++) backing[j] = lds_u32(base + j * kStackStride);
	for (uint32_t a = base + kEvict * kStackStride; a < top; a += kStackStride) sts_u32(a - kEvict * kStackStride, lds_u32(a));
}
__device__ __noinline__ void stack_restore(uint32_t base, const uint32_t* backing) { for (int j = 0; j < kEvict; j++) sts_u32(base + j * kStackStride, backing[j]); }
struct SmemStack {
	uint32_t base, top;  // 32-bit shared-window addresses: s_stack[0][threadIdx.x] and the next free entry; a push or pop is one ST/LD.shared and one add
	int spilled;         // entries in the backing store
	uint32_t* backing;   // [kTraversalStack] in local memory, declared by the kernel
	__device__ __forceinline__ void bind(const uint32_t* slot0, uint32_t* local_backing) { base = top = static_cast<uint32_t>(__cvta_generic_to_shared(slot0)); backing = local_backing; spilled = 0; }
	__device__ __forceinline__ void reset() { top = base; spilled = 0; }
	__device__ __forceinline__ void push(uint32_t v) { sts_u32(top, v); top += kStackStride; }
	__device__ __forceinline__ uint32_t pop() { top -= kStackStride; return lds_u32(top); }
	__device__ __forceinline__ bool empty() const { return top == base; }
	__device__ __forceinline__ void room() {
		if (top > base + (kSmemStack - 3) * kStackStride) { stack_evict(base, top, backing + spilled); spilled += kEvict; top -= kEvict * kStackStride; }
	}
	__device__ __forceinline__ bool refill() {
		if (spilled == 0) return false;
		spilled -= kEvict; stack_restore(base, backing + spilled); top = base + kEvict * kStackStride;
		return true;
	}
};
// The traversal kernels run 32 per-lane walks per warp (b2r_shade.h describes the tree and the per-lane state machines). One
// loop iteration = one wide-node visit for every live lane: the warp stages the lanes' 32 nodes through shared memory
// (warp_stage_nodes); the four slab tests run as one straight-line pass; leaf slots (sphere inlined in the node) are tested
// right away from the staged row; finished lanes are refilled from the warp's pool as soon as fewer than kRefillBelow lanes
// are alive. Results do not depend on any of this: the closest hit is the minimum over every sphere whose ancestors' boxes pass
// (== brute force, ties to the lowest index), any-hit is an order-independent boolean.
// Measured and rejected (round 1, C3): postponing the leaf tests until a dozen lanes hold one ("speculative traversal", spheres
// re-fetched from scene.prims) — 20 % slower, the later culling and the re-fetch cost more than the denser sphere tests save;
// ordering the children with the slot index in the low key bits and min/max pairs — same SASS size as the compare-and-swap
// network (the compiler already emits VIMNMX), 5 % slower; refill thresholds 16/20/28 and 12/20 stack entries in shared memory —
// flat; full-sweep SAH and a cost-optimal 2->4 collapse of the traversal tree — 12.3 instead of 12.4 node visits per ray.
// The loop itself, for a Walk (TravClosestT / TravAnyT over SmemStack) and the kernel's three pieces: read(t, idx) arms the walk with
// claimed ray idx, step(t, row) visits the staged node row and returns false once the ray is finished, write(t, idx) stores its result.
template <class Walk, class Read, class Step, class Write>
__device__ __forceinline__ void lane_walks(const WideNode* __restrict__ wide, uint32_t* cursor, const uint32_t n_in, Read read, Step step, Write write) {
	__shared__ __align__(128) float4 s_nodes[kTravBlock / 32][32 * kNodeRowF4];
	__shared__ uint32_t s_stack[kSmemStack][kTravBlock];
	float4* rows = s_nodes[threadIdx.x >> 5];
	uint32_t backing[kTraversalStack];
	WarpPool pool; Walk t; bool active = false, unsent = false; uint32_t idx = 0;
	t.node = 0u; t.stack.bind(&s_stack[0][threadIdx.x], backing);
	for (;;) {
		// rays that finished since the last refill hand their results over together (dense stores instead of one per finish)
		if (unsent) { write(t, idx); unsent = false; }
		const uint32_t got = pool.take(!active, cursor, n_in);
		if (got != 0xffffffffu) { idx = got; active = true; read(t, idx); }
		uint32_t live = __ballot_sync(0xffffffffu, active);
		if (live == 0u) break;
		do {
			warp_stage_nodes(wide, rows, active ? t.node : 0u);
			if (active && !step(t, rows + lane_id() * kNodeRowF4)) { active = false; unsent = true; }
			live = __ballot_sync(0xffffffffu, active);
		} while (live != 0u && (pool.dry || __popc(live) >= kRefillBelow));
	}
}

// ---- bounce 0: packet traversal ------------------------------------------------------------------------------------------------
// Camera rays are coherent: the 32 consecutive tile-order pixels of a warp (two rows of 16 in one 16x16 tile) walk almost the same
// nodes — measured on C3, ONE walk for the whole warp visits 14.9 nodes per 32 rays where 32 per-lane walks take 14.0 warp-steps. So for
// primary rays the warp walks the tree as a packet: the node is fetched once for the warp (eight broadcast LDG.128: 8 L1 wavefronts
// instead of the ~90 of the staged per-lane fetch), every lane slab-tests the four slots with its own ray, a slot is taken when ANY lane
// passes it within its own best distance (the link is warp-uniform, so leaf / inner is a uniform branch: the sphere test of a leaf slot
// runs once per slot, predicated on the lanes that passed its box), inner slots are ordered by the packet's minimum entry distance
// (REDUX.MIN), and there is ONE stack per warp in shared memory with no per-lane loops at all. Each lane still keeps its own closest
// hit, and a lane only tests spheres whose box its own ray passes, so every lane's result is exactly what its own walk would give.
constexpr int kPacketStack = 64;
// RPL rays per lane: a packet is 32 * RPL consecutive tile-order pixels (RPL = 4: eight rows of 16 = half a 16x16 tile, of one sample). The node
// fetch, the link tests, the ordering network and the stack work are paid once per packet; the slab and sphere tests once per ray (all camera
// rays share the origin, so a ray costs 14 registers). Measured on C3 / C4 (frame time, A/B in one run, frames bit-identical): RPL 1 22.40 ms,
// 2 21.81 (80 registers), 4 21.65 / 197.8 (101 registers), 8 22.72 / 206.3 (162 registers: too few warps left).
#ifndef B2R_PACKET_RPL
#define B2R_PACKET_RPL 4
#endif
// LENS: thin-lens camera rays leave different points of the lens disk, so each ray keeps its own origin (3 more registers per ray). The walk
// stays exact for any rays (each lane keeps its own best and tests only boxes its own ray passes); only coherence changes. RPL 4 with a lens:
// 118 registers, no spills; measured on C3 against RPL 2 (79 registers), A/B in one run: bounce 0 2.92 / 3.03 / 6.58 ms against 3.03 / 3.17 /
// 6.93 ms for circles of confusion of 4, 7.5 and 75 pixels at twice the focus distance (DESIGN §6).
#ifndef B2R_PACKET_RPL_LENS
#define B2R_PACKET_RPL_LENS 4
#endif
template <bool COUNT, int RPL = 1, bool LENS = false>
__global__ void __launch_bounds__(kTravBlock) k_intersect_packet(const Params p, const uint32_t bounce) {
	// The camera rays are GENERATED here (Renderer.hpp:97-127: hash_2d -> PCG -> Camera::generate_ray, in registers) and their path
	// records and zeroed radiance entries written behind the walk (plain coalesced stores that nobody waits for) for k_shade to read:
	// there is no separate ray-generation launch and no read-back of 32 B per ray in front of the traversal.
	const uint32_t n_in = p.batch->n_slots * p.frame.npix;   // a multiple of 256: whole tiles of whole samples
	const float4* __restrict__ wide4 = reinterpret_cast<const float4*>(p.scene.wide);
	__shared__ uint2 s_pstack[kTravBlock / 32][kPacketStack];
	uint2* stack = s_pstack[threadIdx.x >> 5];
	uint32_t c_sphere = 0, c_box = 0;
	uint32_t next = 0, end = 0;
	constexpr uint32_t kClaim = 128u * RPL;  // four packets per claim
	for (;;) {
		if (next >= end) {
			uint32_t b = 0;
			if (lane_id() == 0) b = atomicAdd(p.cnt.work_a + bounce, kClaim);
			b = __shfl_sync(0xffffffffu, b, 0);
			if (b >= n_in) break;
			next = b; end = min(b + kClaim, n_in);
		}
		const uint32_t idx0 = next + lane_id(); next += 32u * RPL;
		constexpr int NO = LENS ? RPL : 1;   // origins kept: one per ray with a lens, one shared by the packet's camera rays without
		float ox[NO], oy[NO], oz[NO], dx[RPL], dy[RPL], dz[RPL], ix[RPL], iy[RPL], iz[RPL], nx[RPL], ny[RPL], nz[RPL], ax[RPL], ay[RPL], az[RPL], best[RPL]; int32_t prim[RPL];
#pragma unroll
		for (int r = 0; r < RPL; r++) {
			const uint32_t idx = idx0 + 32u * r;
			const uint32_t sl = div_by(idx, p.frame.npix, p.frame.npix_magic);
			const PathState s0 = primary_path<LENS>(p.frame, p.batch->cam, p.batch->acc[sl], sl, idx - sl * p.frame.npix, p.batch->lens);
			store_path(p.q, 0, idx, s0); rad_zero(p.rad, p.frame.npix, s0.pid);
			const int ro = LENS ? r : 0;
			ox[ro] = s0.ox; oy[ro] = s0.oy; oz[ro] = s0.oz; dx[r] = s0.dx; dy[r] = s0.dy; dz[r] = s0.dz;   // (without a lens all camera rays leave the same point)
			slab_setup(ox[ro], oy[ro], oz[ro], dx[r], dy[r], dz[r], &ix[r], &iy[r], &iz[r], &nx[r], &ny[r], &nz[r], &ax[r], &ay[r], &az[r]);
			best[r] = FLT_MAX; prim[r] = -1;
		}
		uint32_t node = 0u, sp = 0u;
		for (;;) {
			const float4* nd = wide4 + static_cast<size_t>(node) * 8u;
			float4 na[4], nb[4];
#pragma unroll
			for (int k = 0; k < 4; k++) { na[k] = ldg4(nd + 2 * k); nb[k] = ldg4(nd + 2 * k + 1); }   // the whole node up front: eight broadcast loads in flight (every lane reads the same address)
			uint32_t key[4], link[4];
#pragma unroll
			for (int k = 0; k < 4; k++) {
				const float4 a = na[k], b = nb[k];
				const int32_t l = __float_as_int(b.z);                          // warp-uniform
				key[k] = 0xffffffffu; link[k] = static_cast<uint32_t>(l);
				float tn[RPL]; bool h[RPL]; bool any = false; uint32_t tmin = 0xffffffffu;
#pragma unroll
				for (int r = 0; r < RPL; r++) {
					slab(a, b, ix[r], iy[r], iz[r], nx[r], ny[r], nz[r], ax[r], ay[r], az[r], best[r], &tn[r], &h[r]);  // an empty slot's box (h = -1e30) fails every constrained axis (camera rays keep at least one, slab_setup)
					any = any || h[r]; tmin = min(tmin, h[r] ? __float_as_uint(tn[r]) : 0xffffffffu);
				}
				if (COUNT && l != kEmptyLink) c_box += RPL;
				if (__ballot_sync(0xffffffffu, any) == 0u) continue;
				if (l < 0) {  // leaf slot: the rays that pass its box test the sphere
#pragma unroll
					for (int r = 0; r < RPL; r++) if (h[r]) {
						float d; if (COUNT) c_sphere++;
						const int ro = LENS ? r : 0;
						if (sphere_hit_closest(a.x, a.y, a.z, a.w, ox[ro], oy[ro], oz[ro], dx[r], dy[r], dz[r], &d) && (d < best[r] || (d == best[r] && ~l < prim[r]))) { best[r] = d; prim[r] = ~l; }
					}
				} else key[k] = __reduce_min_sync(0xffffffffu, tmin);  // the packet's entry distance
			}
			float fb = best[0];
#pragma unroll
			for (int r = 1; r < RPL; r++) fb = fmaxf(fb, best[r]);
			const uint32_t far_best = __reduce_max_sync(0xffffffffu, __float_as_uint(fb));  // a node is dead once it lies behind EVERY ray's hit
			B2R_CSWAP(key[0], link[0], key[1], link[1]); B2R_CSWAP(key[2], link[2], key[3], link[3]);
			B2R_CSWAP(key[0], link[0], key[2], link[2]); B2R_CSWAP(key[1], link[1], key[3], link[3]);
			B2R_CSWAP(key[1], link[1], key[2], link[2]);
			if (key[3] <= far_best) { if (lane_id() == 0) stack[sp] = make_uint2(link[3], key[3]); sp++; }   // (a miss key is 0xffffffff > any distance)
			if (key[2] <= far_best) { if (lane_id() == 0) stack[sp] = make_uint2(link[2], key[2]); sp++; }
			if (key[1] <= far_best) { if (lane_id() == 0) stack[sp] = make_uint2(link[1], key[1]); sp++; }
			__syncwarp();
			if (key[0] <= far_best) { node = link[0]; continue; }
			bool found = false;
			while (sp > 0u) {
				const uint2 e = stack[--sp];
				if (e.y <= far_best) { node = e.x; found = true; break; }
			}
			if (!found) break;
		}
#pragma unroll
		for (int r = 0; r < RPL; r++) p.q.H[idx0 + 32u * r] = make_float2(best[r], __int_as_float(prim[r]));
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) { p.cnt.paths[0] = n_in; atomicAdd(p.cnt.stats + ST_EXT, static_cast<unsigned long long>(n_in)); }
	if (COUNT) { stat_add(p.cnt.stats, ST_SPHERE, c_sphere); stat_add(p.cnt.stats, ST_BOX, c_box); }
}

// closest-hit traversal of queue side (bounce & 1). After bounce 0 every path leaves the surface of a sphere, and its walk starts at the
// node holding that sphere (q.N, written by k_shade) and climbs (TravClosestT); camera rays (bounce 0 without the packet kernel) start at
// the root. The walk is exact from any node of the tree it walks, so what a start node must be is an index into that tree: k_shade wrote it
// from the leaf_node table of the same table set, in the same batch — a batch's launches all read one set (the side's own copy, refreshed
// on the side's stream only between its batches, or the primary arrays, which a scene write reaches only in stream order behind the
// batch), and no path outlives its batch.
// (63 registers without a minimum-blocks bound = 8 resident CTAs. Measured: bounding it to 8 costs 4 %; 71/79/96 registers with
// 7/6/5 CTAs cost 3/5/16 %; 56/48 registers with 9/10 CTAs and a shorter shared-memory stack cost 5/8 %.)
template <bool COUNT, bool EXACT, uint32_t TNB>
__global__ void __launch_bounds__(kTravBlock) k_intersect_closest(const Params p, const uint32_t bounce) {
	const uint32_t n_in = p.cnt.paths[bounce];
	const int side = bounce & 1;
	const uint32_t* __restrict__ parent = p.scene.parent;
	uint32_t c_sphere = 0, c_box = 0;
	using Walk = TravClosestT<SmemStack>;
	lane_walks<Walk>(p.scene.wide, p.cnt.work_a + bounce, n_in,
		[&](Walk& t, uint32_t idx) {
			const float4 a = p.q.A[side][idx], b = p.q.B[side][idx];
			bool tail = false;
			if (EXACT && bounce > 0u) {  // B2R_FLAG_REFERENCE_EXACT: scalar-tail formula for the last `active % 8` slots of the ray's stream
				const uint32_t pid_i = __float_as_uint(b.w), stream = (pid_i >> 26) * (p.frame.npix >> 8) + ((pid_i & kPixMask) >> 8);
				tail = static_cast<uint32_t>(p.ex.slot[side][idx]) >= (static_cast<uint32_t>(p.ex.act[side][stream]) & ~7u);
			}
			t.begin(Ray{a.x, a.y, a.z, a.w, b.x, b.y}, tail, bounce == 0u ? 0u : p.q.N[side][idx], parent);
		},
		[&](Walk& t, const float4* row) { return t.template step_staged<COUNT, TNB>(row, p.scene.stack_tn_bits, parent, &c_sphere, &c_box); },
		[&](const Walk& t, uint32_t idx) { p.q.H[idx] = make_float2(t.best, __int_as_float(t.prim)); });
	if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(p.cnt.stats + ST_EXT, static_cast<unsigned long long>(n_in));
	if (COUNT) { stat_add(p.cnt.stats, ST_SPHERE, c_sphere); stat_add(p.cnt.stats, ST_BOX, c_box); }
}
// shade the hit records: light sample -> shadow queue, emission, BRDF sample / roulette -> next path queue.
// Same CTA structure as the brute-force kernel: hits are collected in a shared-memory queue and shaded a full CTA at a time.
template <bool EXACT, bool GGX = false, bool DIELECTRIC = false>
__global__ void __launch_bounds__(kBruteBlock, B2R_SHADE_MIN_BLOCKS) k_shade(const Params p, const uint32_t bounce) {
	constexpr int kQ = 2 * kBruteBlock;
	__shared__ uint32_t s_hit_i[kQ]; __shared__ float s_hit_t[kQ]; __shared__ int32_t s_hit_prim[kQ];
	__shared__ uint32_t s_cnt_a[kBruteWarps], s_cnt_b[kBruteWarps], s_cnt_c[kBruteWarps], s_base, s_sbase;
	const SceneDev& sc = p.scene;
	const uint32_t n_in = p.cnt.paths[bounce];
	const int side = bounce & 1;
	const bool mis = !(p.frame.flags & B2R_FLAG_NO_MIS);
	const bool last = bounce + 1 >= p.frame.max_bounces;
	uint32_t c_hits = 0, c_term = 0, c_drop = 0, c_events = 0, c_inline_shadow = 0;
	if (blockIdx.x * kBruteBlock >= n_in) return;
	uint32_t queued = 0, base = blockIdx.x * kBruteBlock;
	for (;;) {
		const bool more = base < n_in;
		if (more) {
			const uint32_t i = base + threadIdx.x;
			const bool live = i < n_in;
			float depth = FLT_MAX; int32_t prim = -1;
			if (live) { const float2 h = p.q.H[i]; depth = h.x; prim = __float_as_int(h.y); }
			const bool is_hit = live && prim >= 0;
#ifndef B2R_NO_SHADE_PREFETCH
			// what the shading phase will read for this hit — its path record (44 B over five planes), its sphere and material id — is asked for
			// now, before the hits are compacted behind two barriers: the shading phase's dependent round trips then hit in L1
			if (is_hit) {
				prefetch_l1(p.q.A[side] + i); prefetch_l1(p.q.B[side] + i); prefetch_l1(p.q.T[side] + i); prefetch_l1(p.q.T[side] + p.q.cap + i); prefetch_l1(p.q.T[side] + 2u * p.q.cap + i);
				prefetch_l1(sc.prims + prim); prefetch_l1(sc.prim_mat + prim); prefetch_l1(sc.leaf_node + prim);
			}
			if (base + gridDim.x * kBruteBlock + threadIdx.x < n_in) prefetch_l1(p.q.H + base + gridDim.x * kBruteBlock + threadIdx.x);  // the next chunk's hit records
#endif
			if (live && !is_hit) {  // miss shader (Renderer.hpp:408-420)
				c_term++;
				if (sc.has_ambient) { const PathState sm = load_path(p.q, side, i); rad_add(p.rad, p.frame.npix, sm.pid, shade_sky(sc, sm), f3{0.0f, 0.0f, 0.0f}, true, false); c_events++; }
			}
			uint32_t n_hits;
			const uint32_t slot = queued + block_rank(is_hit, s_cnt_a, &n_hits);
			if (is_hit) { s_hit_i[slot] = i; s_hit_t[slot] = depth; s_hit_prim[slot] = prim; }
			queued += n_hits;
			base += gridDim.x * kBruteBlock;
			__syncthreads();
		}
		if (queued < static_cast<uint32_t>(kBruteBlock) && more) continue;
		if (queued == 0) break;
		const uint32_t take = min(queued, static_cast<uint32_t>(kBruteBlock));
		const uint32_t qi = queued - take + threadIdx.x;
		const bool shade = threadIdx.x < take;
		queued -= take;
		bool keep = false, want_shadow = false; ShadowRay sr; PathState s; uint32_t pid = 0, ex_slot = 0, ex_mat = 0, start = 0;
		if (shade) {
			const uint32_t hi = s_hit_i[qi]; const float depth = s_hit_t[qi]; const int32_t prim = s_hit_prim[qi];
			start = __ldg(sc.leaf_node + prim);  // where this hit's shadow ray and continued path will start their walks (asked for early: nothing waits for it before the queue writes)
			s = load_path(p.q, side, hi); pid = s.pid;
			if (EXACT) ex_slot = bounce == 0u ? (pid & 255u) : static_cast<uint32_t>(p.ex.slot[side][hi]);  // bounce 0: slot = pixel ID
			const uint32_t acc = p.batch->acc[s.pid >> 26], seed = pixel_seed(s.pid & kPixMask, p.frame.max_bounces);
			const Surface sf = shade_surface<GGX, DIELECTRIC>(sc, s, depth, prim, p.mat_diel);
			if (EXACT) ex_mat = static_cast<uint32_t>(sf.mat);
			c_hits++;
			if (last) { rad_zero(p.rad, p.frame.npix, s.pid); c_drop++; }  // Q11
			else {
				if (mis) want_shadow = shade_light_sample<GGX, DIELECTRIC>(sc, sf, s, prim, acc, seed, bounce, &sr);
				if (sf.emissive) {
					// the reference adds the light sample first, then the emission (Renderer.hpp:304-353). For the (rare) emissive hit
					// that also has a shadow ray the any-hit traversal is done right here so that order holds; every other shadow ray
					// goes to the shadow queue and is traced by k_intersect_shadow.
					const f3 emit = shade_emission<DIELECTRIC>(sc, sf, s, depth, bounce, mis);
					if (want_shadow) {
						uint32_t cs = 0, cb = 0;
						const bool occluded = traverse_any<false>(sc.wide, Ray{sr.o.x, sr.o.y, sr.o.z, sr.d.x, sr.d.y, sr.d.z}, sr.tfar, &cs, &cb, sc.parent, 0u);
						rad_add(p.rad, p.frame.npix, s.pid, sr.L, emit, !occluded, true);
						want_shadow = false; c_inline_shadow++;
					} else rad_add(p.rad, p.frame.npix, s.pid, emit, f3{0.0f, 0.0f, 0.0f}, true, false);
					c_events++;
				}
				keep = shade_continue<GGX, DIELECTRIC>(sf, &s, acc, seed, bounce);
				if (!keep) c_term++;
			}
		}
		uint32_t n_shadow, n_keep, srank, rank;
		block_rank2(want_shadow, keep, s_cnt_b, s_cnt_c, &srank, &n_shadow, &rank, &n_keep);  // barrier: queue reads above are done before the next phase 1 writes
		if (threadIdx.x == 0) {
			s_sbase = n_shadow ? atomicAdd(p.cnt.shadow + bounce, n_shadow) : 0u;
			s_base = n_keep ? atomicAdd(p.cnt.paths + bounce + 1, n_keep) : 0u;
		}
		__syncthreads();
		if (want_shadow) {
			const uint32_t d = s_sbase + srank;
			p.q.SA[d] = make_float4(sr.o.x, sr.o.y, sr.o.z, sr.d.x);
			p.q.SB[d] = make_float4(sr.d.y, sr.d.z, sr.tfar, __uint_as_float(pid));
			p.q.SL[d] = sr.L.x; p.q.SL[p.q.cap + d] = sr.L.y; p.q.SL[2u * p.q.cap + d] = sr.L.z;
			p.q.SS[d] = start;
		}
		if (keep) {
			store_path(p.q, side ^ 1, s_base + rank, s);
			p.q.N[side ^ 1][s_base + rank] = start;
			if (EXACT) {  // (stream, slot) -> material and next-queue index, for k_stream_rank
				const uint32_t e = (pid >> 26) * p.frame.npix + ((pid & kPixMask) & ~255u) + ex_slot;
				p.ex.key[e] = static_cast<uint8_t>(ex_mat + 1u); p.ex.next_idx[e] = s_base + rank;
			}
		}
	}
	stat_add(p.cnt.stats, ST_HITS, c_hits); stat_add(p.cnt.stats, ST_TERM, c_term);
	stat_add(p.cnt.stats, ST_DROPPED, c_drop); stat_add(p.cnt.stats, ST_EVENTS, c_events); stat_add(p.cnt.stats, ST_SHADOW, c_inline_shadow);
}
// shadow rays of this bounce: the climbing any-hit walk (TravAnyT) from the node that holds each ray's origin sphere; unoccluded light
// samples are added to the pixel's radiance.
template <bool COUNT>
__global__ void __launch_bounds__(kTravBlock, 8) k_intersect_shadow(const Params p, const uint32_t bounce) {
	const uint32_t n_in = p.cnt.shadow[bounce];
	const uint32_t* __restrict__ parent = p.scene.parent;
	uint32_t c_sphere = 0, c_box = 0, c_events = 0, pid = 0;
	using Walk = TravAnyT<SmemStack>;
	lane_walks<Walk>(p.scene.wide, p.cnt.work_b + bounce, n_in,
		[&](Walk& t, uint32_t idx) {
			const float4 a = p.q.SA[idx], b = p.q.SB[idx];
			pid = __float_as_uint(b.w);
			t.begin(Ray{a.x, a.y, a.z, a.w, b.x, b.y}, b.z, p.q.SS[idx], parent);
		},
		[&](Walk& t, const float4* row) { return t.template step_staged<COUNT>(row, parent, &c_sphere, &c_box); },
		[&](const Walk& t, uint32_t idx) {
			if (t.occluded) return;  // the light sample is dropped
			const f3 L{p.q.SL[idx], p.q.SL[p.q.cap + idx], p.q.SL[2u * p.q.cap + idx]};
			rad_add(p.rad, p.frame.npix, pid, L, f3{0.0f, 0.0f, 0.0f}, true, false); c_events++;
		});
	if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(p.cnt.stats + ST_SHADOW, static_cast<unsigned long long>(n_in));
	stat_add(p.cnt.stats, ST_EVENTS, c_events);
	if (COUNT) { stat_add(p.cnt.stats, ST_SPHERE, c_sphere); stat_add(p.cnt.stats, ST_BOX, c_box); }
}


// ---------------------------------------------------------------------------------------------- accumulate + resolve
// Fold the batch's per-sample radiance into its median-of-means bucket, in sample order (Renderer.hpp:424-430 adds one
// sample at a time; bucket = acc % K, :82). RAD is not cleared here: the primary-ray stage of the next batch starts every
// (sample, pixel) entry at 0 with a plain store, which halves this kernel's HBM traffic.
__global__ void __launch_bounds__(kBlock) k_accumulate(const Params p) {
	__shared__ uint32_t s_order[kMaxSlots];   // slots grouped by bucket, increasing sample index inside a bucket
	__shared__ uint32_t s_first[kMaxSlots + 1];  // group boundaries per bucket (buckets <= 64)
	const uint32_t npix4 = p.frame.npix / 4u, n = 3u * npix4, slots = p.batch->n_slots, K = p.frame.buckets;
	if (threadIdx.x == 0) {
		uint32_t m = 0;
		const unsigned long long fold = p.batch->fold;
		for (uint32_t k = 0; k < K; k++) { s_first[k] = m; for (uint32_t s = 0; s < slots; s++) if (((fold >> s) & 1ull) && p.batch->acc[s] % K == k) s_order[m++] = s; }
		s_first[K] = m;
	}
	__syncthreads();
	const float4* __restrict__ rad = reinterpret_cast<const float4*>(p.rad); float4* __restrict__ acc = reinterpret_cast<float4*>(p.acc);
	const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const uint32_t c = i / npix4, t4 = i - c * npix4;
		for (uint32_t k = 0; k < K; k++) {
			const uint32_t b0 = s_first[k], b1 = s_first[k + 1];
			if (b0 == b1) continue;
			float4* dst = acc + (static_cast<size_t>(k) * 3u + c) * npix4 + t4;
			float4 sum = *dst;
			for (uint32_t j = b0; j < b1; j += 4u) {  // four independent loads in flight, added in sample order
				float4 v[4];
#pragma unroll
				for (uint32_t u = 0; u < 4u; u++) v[u] = (j + u < b1) ? rad[(static_cast<size_t>(s_order[j + u]) * 3u + c) * npix4 + t4] : zero;
#pragma unroll
				for (uint32_t u = 0; u < 4u; u++) if (j + u < b1) { sum.x += v[u].x; sum.y += v[u].y; sum.z += v[u].z; sum.w += v[u].w; }
			}
			*dst = sum;
		}
	}
}
// median of K bucket sums. K == 5 is the reference's network (Sampling.hpp:13-21); other K are this repo's definition:
// odd K -> middle order statistic, even K -> mean of the two middle ones (SURVEY §8d, C2).
// where each bucket's [3][npix] sums live: this GPU's accumulator, or — multi-GPU — the owner's HBM mapped over NVLink
struct BucketPtrs { const float* k[64]; };
__device__ __forceinline__ float median_buckets_at(const BucketPtrs& bp, uint32_t K, uint32_t off) {
	if (K == 5) return median_of_5(bp.k[0][off], bp.k[1][off], bp.k[2][off], bp.k[3][off], bp.k[4][off]);
	if (K == 3) return median_of_3(bp.k[0][off], bp.k[1][off], bp.k[2][off]);
	if (K == 1) return bp.k[0][off];
	if (K == 8) return median_of_8(bp.k[0][off], bp.k[1][off], bp.k[2][off], bp.k[3][off], bp.k[4][off], bp.k[5][off], bp.k[6][off], bp.k[7][off]);
	float v[64];
	for (uint32_t k = 0; k < K; k++) {  // insertion sort
		float x = bp.k[k][off]; int j = static_cast<int>(k) - 1;
		while (j >= 0 && v[j] > x) { v[j + 1] = v[j]; j--; }
		v[j + 1] = x;
	}
	return (K & 1u) ? v[K / 2u] : (v[K / 2u - 1u] + v[K / 2u]) * 0.5f;
}
// Renderer::Render, Renderer.hpp:436-478: one thread per pixel (tile order in, raster RGBA out). With peer pointers this one
// kernel is the whole multi-GPU combine: the median network pulls each bucket from its owner over NVLink (coalesced 128-byte
// peer loads) — no all-reduce, no staging copy.
__global__ void __launch_bounds__(kBlock) k_resolve(const FrameDev frame, const __grid_constant__ BucketPtrs bp, float4* __restrict__ fb, const float scale, const int tonemap,
                                                    const uint32_t t_begin, const uint32_t t_end) {
	const uint32_t npix = frame.npix, K = frame.buckets;
	for (uint32_t t = t_begin + blockIdx.x * blockDim.x + threadIdx.x; t < t_end; t += gridDim.x * blockDim.x) {
		float r = scale * median_buckets_at(bp, K, t);
		float g = scale * median_buckets_at(bp, K, npix + t);
		float b = scale * median_buckets_at(bp, K, 2u * npix + t);
		if (tonemap) aces_tonemap(&r, &g, &b);
		int32_t x, y; pixel_xy(t, frame, &x, &y);
		fb[static_cast<size_t>(y) * frame.width + x] = make_float4(r, g, b, 1.0f);
	}
}

// ---------------------------------------------------------------------------------------------- multi-GPU team: device-side hand-shakes
// One TeamSync block per rank, in its own HBM, mapped by every peer (CUDA IPC). A rank announces an event by storing the frame number
// into ITS entry of every peer's block (release, system scope, over NVLink); a rank waits by spinning on its own block (acquire, local
// HBM). Frame numbers only grow, so nothing is ever reset. Every signal is enqueued on the signalling rank's stream before anything
// that rank waits for, so the waits cannot deadlock; they still give up after kTeamSpinLimit cycles and flag an error instead of hanging
// the GPU if a peer died.
constexpr int kTeamMax = 16;
struct TeamSync {
	uint32_t ready[kTeamMax];   // ready[r]  = last frame whose buckets rank r has finished accumulating
	uint32_t done[kTeamMax];    // done[r]   = last frame rank r has finished resolving (its reads of peer buckets and its slab writes are complete)
	uint32_t copied;            // last frame rank 0 has copied out of its framebuffer (the framebuffer may be overwritten)
	uint32_t error;             // non-zero: a wait timed out
};
struct TeamPeers { TeamSync* sync[kTeamMax]; };
enum TeamField { TEAM_READY = 0, TEAM_DONE = 1, TEAM_COPIED = 2 };
constexpr long long kTeamSpinLimit = 8000000000ll;  // ~4 s at 1.9 GHz
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__global__ void k_team_signal(const __grid_constant__ TeamPeers peers, const uint32_t n_ranks, const uint32_t my_rank, const int field, const uint32_t frame) {
	const uint32_t r = threadIdx.x;
	if (r >= n_ranks) return;
	__threadfence_system();  // everything this rank wrote before (stream order) is visible system-wide before the flag is
	TeamSync* s = peers.sync[r];
	st_release_sys(field == TEAM_READY ? &s->ready[my_rank] : field == TEAM_DONE ? &s->done[my_rank] : &s->copied, frame);
}
__global__ void k_team_wait(TeamSync* mine, const uint32_t n_ranks, const int field, const uint32_t frame) {
	const uint32_t r = threadIdx.x;
	if (r >= (field == TEAM_COPIED ? 1u : n_ranks)) return;
	const uint32_t* flag = field == TEAM_READY ? &mine->ready[r] : field == TEAM_DONE ? &mine->done[r] : &mine->copied;
	const long long t0 = clock64();
	while (static_cast<int32_t>(ld_acquire_sys(flag) - frame) < 0) {
		if (clock64() - t0 > kTeamSpinLimit) { atomicExch(&mine->error, 1u + static_cast<uint32_t>(field)); break; }
		__nanosleep(200);
	}
}

// ---------------------------------------------------------------------------------------------- scene edit: refit
// Application.cpp:508-509 rebuilds the BVH on every geometry drag. Here the traversal tree keeps its topology and only its boxes
// are recomputed, on the GPU, from the moved spheres: one launch per BFS level, deepest first (children always sit on a deeper
// level), four threads per 128-byte node = one per slot (refit_slot, b2r_shade.h; shared with the host twin the tests compare with).
__global__ void __launch_bounds__(kBlock) k_refit_level(float4* __restrict__ wide, const float4* __restrict__ prims, const uint32_t* __restrict__ remap, const OriginBox ob, const uint32_t first, const uint32_t count) {
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < count * 4u) refit_slot(wide, prims, remap, ob, first + (i >> 2), static_cast<int>(i & 3u));
}
// parent[] and leaf_node[] of the device tree as it stands (after an upload, a refit that re-linked leaves, or a device build): one thread per slot
__global__ void __launch_bounds__(kBlock) k_link_tables(const float4* __restrict__ wide, const uint32_t n_nodes, uint32_t* __restrict__ parent, uint32_t* __restrict__ leaf_node) {
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, node = i >> 2;
	if (node >= n_nodes) return;
	if (i == 0u) parent[0] = 0u;
	const int32_t l = __float_as_int(wide[static_cast<size_t>(i) * 2u + 1u].z);
	if (l == kEmptyLink) return;
	if (l < 0) leaf_node[~l] = node; else parent[l] = node;
}
// ---------------------------------------------------------------------------------------------- GPU tree build (B2R_FLAG_GPU_TREE)
// The traversal tree built on the device for edits that add or remove spheres (the reference rebuilds its BVH on every edit,
// Application.cpp:508-509): 30-bit curve keys of the sphere centres (the Hilbert index of the centre's cell, b2r_shade.h morton_key — a run of
// consecutive Hilbert keys is a connected set of cells, a Z-curve run is not), a stable radix sort (CUB), then an implicit, perfectly balanced
// 4-ary topology over the sorted order — four spheres to a bottom node, four nodes to a parent — whose links follow from the sphere count
// alone (k_packed_links), and the boxes from the same k_refit_level passes a scene edit uses. Results do not depend on the tree; its
// quality does: on C3's overlapping spheres it needs ~2x the node visits of the host's SAH tree (4x when it sorted by Morton code; DESIGN.md),
// so it is the instant tree after an edit, not the default; the sweep tree below (B2R_FLAG_GPU_SAH) is the better one. Host twin: build_packed_tree (b2r_host.cpp); the tests compare the two bit for bit.
struct PackedLevels { uint32_t first[24]; uint32_t levels; };   // level_first of packed_levels(): root level first
__global__ void __launch_bounds__(kBlock) k_morton_keys(const float4* __restrict__ prims, const uint32_t n, const float lo0, const float lo1, const float lo2,
                                                        const float s0, const float s1, const float s2, uint32_t* __restrict__ keys, uint32_t* __restrict__ idx) {
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float lo[3] = {lo0, lo1, lo2}, scale[3] = {s0, s1, s2};
	const float4 p = prims[i];
	keys[i] = morton_key(p.x, p.y, p.z, lo, scale); idx[i] = i;
}
__global__ void __launch_bounds__(kBlock) k_packed_links(float4* __restrict__ wide, const __grid_constant__ PackedLevels lv, const uint32_t n, const uint32_t* __restrict__ order) {
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, node = t >> 2, k = t & 3u;
	if (node >= lv.first[lv.levels]) return;
	uint32_t l = 0; while (node >= lv.first[l + 1]) l++;
	const bool bottom = l + 1 == lv.levels;
	const uint32_t i = node - lv.first[l], c = 4u * i + k;
	const uint32_t child_count = bottom ? n : lv.first[l + 2] - lv.first[l + 1];
	float4* slot = wide + static_cast<size_t>(node) * 8 + 2 * k;
	if (c >= child_count) { slot[0] = make_float4(0.0f, 0.0f, 0.0f, 0.0f); slot[1] = make_float4(-1.0e30f, -1.0e30f, __int_as_float(kEmptyLink), -1.0e30f); }
	else { slot[0] = make_float4(0.0f, 0.0f, 0.0f, 0.0f); slot[1] = make_float4(0.0f, 0.0f, __int_as_float(bottom ? ~static_cast<int32_t>(order[c]) : static_cast<int32_t>(lv.first[l + 1] + c)), 0.0f); }
}
// ---- sweep build (B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH; host twin build_sweep_tree, shared arithmetic b2r_shade.h sweep_*). The spheres stay
// in curve order (the radix sort above); `head[p]` says that position p starts a run. One opening round = two segmented inclusive scans of the
// sphere boxes (operator sweep_join: fwd[p] = box of [run start, p], bwd[p] = box of [p, run end)), every possible cut of every run costed
// from them and the cheapest filed under the run's start with an atomic minimum (k_sweep_tiles / k_sweep_carry / k_sweep_cuts below), then
// k_sweep_open (one thread per node of the level: cut the run with the largest box; the third round also counts the node's runs of two or
// more spheres). Three rounds make a node's four runs; an exclusive sum of the counts and k_sweep_emit then write the level's links and the
// next level's nodes (15 launches per level). The host reads one count per level (how many nodes the next level has).
__global__ void __launch_bounds__(kBlock) k_sweep_boxes(const float4* __restrict__ prims, const uint32_t* __restrict__ order, const uint32_t n, SweepItem* __restrict__ box, uint32_t* __restrict__ head, SweepKids* __restrict__ root) {
	const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
	if (p >= n) return;
	SweepItem it; sweep_sphere_box(prims[order[p]], &it);
	box[p] = it; head[p] = p == 0u ? 1u : 0u;
	if (p == 0u) { SweepKids K; for (int k = 0; k < 4; k++) { K.a[k] = 0u; K.b[k] = 0u; } K.b[0] = n; K.n = 1u; *root = K; }   // the root node: one run, everything
}
// The segmented scans, hand-written for this item (a 24-byte box + run bookkeeping) and fused with what produces and consumes them, so that
// no scanned array ever reaches memory: a tile is kSweepTile consecutive positions = one block.
//   k_sweep_tiles  the join of each tile's items, forwards and backwards (2 x 32 B per tile); also resets cut_of
//   k_sweep_carry  block 0 / block 1: exclusive scan of the tile joins from the left / from the right = what enters each tile
//   k_sweep_cuts   each tile again: both inclusive scans in shared memory (warp shuffles, then the carried-in item), every cut costed,
//                  the cheapest of a run filed under its first position
// (cub::DeviceScan over materialised items took 35 us per round at 100k spheres against 3 x ~5 us for these.)
constexpr uint32_t kSweepTile = 256u;
__device__ __forceinline__ SweepItem sweep_nothing() { SweepItem e; e.lo0 = e.lo1 = e.lo2 = FLT_MAX; e.hi0 = e.hi1 = e.hi2 = -FLT_MAX; e.pos = 0u; e.flag = 0u; return e; }   // past the end of the array: joins to nothing
// position p as an item of the forward sequence (a run's first position is a segment head and carries the run's start) or of the backward
// one (a run's last position is the head and carries the run's end)
// (`order`: null = the boxes are stored in position order (curve sweep); else position p holds sphere order[p] (three-axis sweep: one order per axis))
__device__ __forceinline__ SweepItem sweep_item(const SweepItem* __restrict__ box, const uint32_t* __restrict__ order, const uint32_t* __restrict__ head, const uint32_t n, const uint32_t p, const bool backward) {
	if (p >= n) return sweep_nothing();
	SweepItem it = box[order ? order[p] : p];
	if (!backward) { it.pos = p; it.flag = head[p]; }
	else { it.pos = p + 1u; it.flag = (p + 1u == n || head[p + 1u] != 0u) ? 1u : 0u; }
	return it;
}
__device__ __forceinline__ SweepItem sweep_shfl_up(const SweepItem& v, const int o) {
	SweepItem r;
	r.lo0 = __shfl_up_sync(0xffffffffu, v.lo0, o); r.lo1 = __shfl_up_sync(0xffffffffu, v.lo1, o); r.lo2 = __shfl_up_sync(0xffffffffu, v.lo2, o); r.pos = __shfl_up_sync(0xffffffffu, v.pos, o);
	r.hi0 = __shfl_up_sync(0xffffffffu, v.hi0, o); r.hi1 = __shfl_up_sync(0xffffffffu, v.hi1, o); r.hi2 = __shfl_up_sync(0xffffffffu, v.hi2, o); r.flag = __shfl_up_sync(0xffffffffu, v.flag, o);
	return r;
}
// inclusive scan (operator sweep_join) of one item per thread in thread order over a block of kSweepTile threads; s_warp: kSweepTile / 32 items.
// Every thread must call it; *total (may be null) receives the join of all items in every thread.
__device__ __forceinline__ SweepItem sweep_block_scan(SweepItem v, SweepItem* s_warp, SweepItem* total) {
	const uint32_t lane = lane_id(), w = threadIdx.x >> 5;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) { const SweepItem u = sweep_shfl_up(v, o); if (lane >= static_cast<uint32_t>(o)) v = sweep_join(u, v); }
	__syncthreads();                      // (s_warp may still be read by a previous call)
	if (lane == 31u) s_warp[w] = v;
	__syncthreads();
	if (w > 0u) { SweepItem pre = s_warp[0]; for (uint32_t k = 1; k < w; k++) pre = sweep_join(pre, s_warp[k]); v = sweep_join(pre, v); }
	if (total) { SweepItem t = s_warp[0]; for (uint32_t k = 1; k < kSweepTile / 32u; k++) t = sweep_join(t, s_warp[k]); *total = t; }
	return v;
}
__global__ void __launch_bounds__(kSweepTile) k_sweep_tiles(const SweepItem* __restrict__ box, const uint32_t* __restrict__ order, const uint32_t* __restrict__ head, const uint32_t n, SweepItem* __restrict__ tile_f, SweepItem* __restrict__ tile_b,
                                                            unsigned long long* __restrict__ cut_of /*null: keep (a later axis of the same round)*/) {
	__shared__ SweepItem s_warp[kSweepTile / 32u];
	const uint32_t t0 = blockIdx.x * kSweepTile, i = threadIdx.x;
	if (cut_of && t0 + i < n) cut_of[t0 + i] = ~0ull;
	SweepItem tf, tb;
	sweep_block_scan(sweep_item(box, order, head, n, t0 + i, false), s_warp, &tf);
	sweep_block_scan(sweep_item(box, order, head, n, t0 + (kSweepTile - 1u - i), true), s_warp, &tb);   // thread order = descending positions
	if (i == 0u) { tile_f[blockIdx.x] = tf; tile_b[blockIdx.x] = tb; }
}
// carry_f[t] = join of tiles 0 .. t-1 in ascending order (t >= 1), carry_b[t] = join of tiles T-1 .. t+1 in descending order (t <= T-2)
__global__ void __launch_bounds__(kSweepTile) k_sweep_carry(const SweepItem* __restrict__ tile_f, const SweepItem* __restrict__ tile_b, const uint32_t tiles, SweepItem* __restrict__ carry_f, SweepItem* __restrict__ carry_b) {
	__shared__ SweepItem s_warp[kSweepTile / 32u];
	__shared__ SweepItem s_part[kSweepTile];
	const bool backward = blockIdx.x == 1u;
	const SweepItem* in = backward ? tile_b : tile_f; SweepItem* out = backward ? carry_b : carry_f;
	const uint32_t chunk = (tiles + kSweepTile - 1u) / kSweepTile, j0 = threadIdx.x * chunk;   // this thread's stretch of the sequence
	auto tile_of = [&](uint32_t j) { return backward ? tiles - 1u - j : j; };
	SweepItem mine = sweep_nothing(); bool any = false;
	for (uint32_t j = j0; j < j0 + chunk && j < tiles; j++) { const SweepItem v = in[tile_of(j)]; mine = any ? sweep_join(mine, v) : v; any = true; }
	s_part[threadIdx.x] = sweep_block_scan(mine, s_warp, nullptr);   // (stretches past the end hold `nothing` and come last)
	__syncthreads();
	SweepItem run = threadIdx.x ? s_part[threadIdx.x - 1u] : sweep_nothing(); bool have = threadIdx.x != 0u;
	for (uint32_t j = j0; j < j0 + chunk && j < tiles; j++) {
		if (have) out[tile_of(j)] = run;
		const SweepItem v = in[tile_of(j)]; run = have ? sweep_join(run, v) : v; have = true;
	}
}
__global__ void __launch_bounds__(kSweepTile) k_sweep_cuts(const SweepItem* __restrict__ box, const uint32_t* __restrict__ order, const uint32_t* __restrict__ head, const uint32_t n, const SweepItem* __restrict__ carry_f, const SweepItem* __restrict__ carry_b,
                                                           unsigned long long* __restrict__ cut_of, float* __restrict__ area_of, const uint32_t axis /*0xffffffff: curve sweep (key = sweep_key)*/, uint32_t* __restrict__ start_of /*may be null*/) {
	__shared__ SweepItem s_warp[kSweepTile / 32u];
	__shared__ SweepItem s_f[kSweepTile], s_b[kSweepTile];   // by position within the tile: box of [run start, p] / of [p, run end)
	const uint32_t tile = blockIdx.x, t0 = tile * kSweepTile, i = threadIdx.x, p = t0 + i;
	{
		SweepItem f = sweep_block_scan(sweep_item(box, order, head, n, p, false), s_warp, nullptr);
		if (tile > 0u) f = sweep_join(carry_f[tile], f);
		s_f[i] = f;
		SweepItem b = sweep_block_scan(sweep_item(box, order, head, n, t0 + (kSweepTile - 1u - i), true), s_warp, nullptr);
		if (tile + 1u < gridDim.x) b = sweep_join(carry_b[tile], b);
		s_b[kSweepTile - 1u - i] = b;
	}
	__syncthreads();
	unsigned long long key = ~0ull; uint32_t start = 0xffffffffu;
	if (p < n) {
		const SweepItem f = s_f[i], b = s_b[i];
		start = f.pos; const uint32_t end = b.pos;
		if (head[p] == 0u) {   // cut in front of p: [start, p) | [p, end); position 0 is a head, so p - 1 exists
			const SweepItem left = i ? s_f[i - 1u] : carry_f[tile];
			key = axis == 0xffffffffu ? sweep_key(sweep_area(left), p - start, sweep_area(b), end - p, p) : sweep_key3(sweep_area(left), p - start, sweep_area(b), end - p, p, axis);
		}
		if (p + 1u == end) area_of[start] = sweep_area(f);
		if (start_of) start_of[p] = start;
	}
	// one atomic per warp while the whole warp sits in one run (the top of the tree), one per lane otherwise
	const uint32_t s0 = __shfl_sync(0xffffffffu, start, 0);
	if (__all_sync(0xffffffffu, start == s0 || p >= n)) {
		for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o); key = other < key ? other : key; }
		if (lane_id() == 0u && key != ~0ull) atomicMin(cut_of + s0, key);
	} else if (key != ~0ull) atomicMin(cut_of + start, key);
}
__global__ void __launch_bounds__(kBlock) k_sweep_open(SweepKids* __restrict__ kids, const uint32_t m, const unsigned long long* __restrict__ cut_of, const float* __restrict__ area_of, uint32_t* __restrict__ head,
                                                       uint32_t* __restrict__ inner /*last round of a level: [m + 1] counts of runs that become nodes; else null*/) {
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > m) return;
	if (j == m) { if (inner) inner[m] = 0u; return; }   // the exclusive sum leaves the level's total there
	SweepKids K = kids[j];
	const uint32_t pos = sweep_open(K, cut_of, area_of);
	if (pos) { kids[j] = K; head[pos] = 1u; }
	if (inner) { uint32_t ni = 0u; for (uint32_t k = 0; k < K.n; k++) ni += (K.b[k] - K.a[k] >= 2u) ? 1u : 0u; inner[j] = ni; }
}
__global__ void __launch_bounds__(kBlock) k_sweep_emit(const SweepKids* __restrict__ kids, const uint32_t m, const uint32_t* __restrict__ inner_before, const uint32_t* __restrict__ order,
                                                       float4* __restrict__ wide, const uint32_t level_first, const uint32_t child_level_first, SweepKids* __restrict__ next_kids) {
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= m) return;
	const SweepKids K = kids[j];
	int32_t link[4]; uint32_t ca[4], cb[4];
	const uint32_t before = inner_before[j];
	const uint32_t ni = sweep_links(K, order, child_level_first + before, link, ca, cb);
	for (uint32_t i = 0; i < ni; i++) { SweepKids C; for (int k = 0; k < 4; k++) { C.a[k] = 0u; C.b[k] = 0u; } C.a[0] = ca[i]; C.b[0] = cb[i]; C.n = 1u; next_kids[before + i] = C; }   // the next level's nodes, one run each
	float4* node = wide + static_cast<size_t>(level_first + j) * 8;
	for (int k = 0; k < 4; k++) {
		node[2 * k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
		node[2 * k + 1] = link[k] == kEmptyLink ? make_float4(-1.0e30f, -1.0e30f, __int_as_float(kEmptyLink), -1.0e30f) : make_float4(0.0f, 0.0f, __int_as_float(link[k]), 0.0f);
	}
}
// ---- three-axis sweep (B2R_FLAG_GPU_SAH3; host twin build_sweep3_tree): three orders of the spheres (sorted by centre x, y, z: ord[axis * n + p]),
// every run the same index range of all three. A round surveys the runs once per axis (the kernels above with `order` and `axis`; the atomic
// minimum then also picks the axis), k_sweep3_open cuts the largest run of every node and notes (tag, position, axis) under the run's start,
// k_sweep3_mark says for every sphere of a cut run whether it goes right, and the three orders are partitioned to match, stably: an exclusive
// sum over "goes left" flags of all 3n entries (CUB) gives every entry its place (k_sweep3_flags / k_sweep3_scatter).
__global__ void __launch_bounds__(kBlock) k_sweep3_boxes(const float4* __restrict__ prims, const uint32_t n, SweepItem* __restrict__ box, uint32_t* __restrict__ keys /*[3n]*/, uint32_t* __restrict__ ids /*[3n]*/,
                                                         uint32_t* __restrict__ head, uint32_t* __restrict__ split_tag, SweepKids* __restrict__ root) {
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float4 s = prims[i];
	SweepItem it; sweep_sphere_box(s, &it); box[i] = it;
	keys[i] = float_order_key(s.x); keys[n + i] = float_order_key(s.y); keys[2u * n + i] = float_order_key(s.z);
	ids[i] = i; ids[n + i] = i; ids[2u * n + i] = i;
	head[i] = i == 0u ? 1u : 0u; split_tag[i] = 0u;
	if (i == 0u) { SweepKids K; for (int k = 0; k < 4; k++) { K.a[k] = 0u; K.b[k] = 0u; } K.b[0] = n; K.n = 1u; *root = K; }
}
__global__ void __launch_bounds__(kBlock) k_sweep3_open(SweepKids* __restrict__ kids, const uint32_t m, const unsigned long long* __restrict__ cut_of, const float* __restrict__ area_of, uint32_t* __restrict__ head,
                                                        uint32_t* __restrict__ split_tag, uint32_t* __restrict__ split_pos, uint32_t* __restrict__ split_axis, const uint32_t tag, uint32_t* __restrict__ inner) {
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > m) return;
	if (j == m) { if (inner) inner[m] = 0u; return; }
	SweepKids K = kids[j];
	uint32_t axis = 0u, a = 0u, b = 0u;
	const uint32_t pos = sweep_open3(K, cut_of, area_of, &axis, &a, &b);
	if (pos) { kids[j] = K; head[pos] = 1u; split_tag[a] = tag; split_pos[a] = pos; split_axis[a] = axis; }
	if (inner) { uint32_t ni = 0u; for (uint32_t k = 0; k < K.n; k++) ni += (K.b[k] - K.a[k] >= 2u) ? 1u : 0u; inner[j] = ni; }
}
__global__ void __launch_bounds__(kBlock) k_sweep3_mark(const uint32_t* __restrict__ ord, const uint32_t n, const uint32_t* __restrict__ start_of, const uint32_t* __restrict__ split_tag, const uint32_t* __restrict__ split_pos,
                                                        const uint32_t* __restrict__ split_axis, const uint32_t tag, uint32_t* __restrict__ right) {
	const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
	if (p >= n) return;
	const uint32_t s = start_of[p];
	if (split_tag[s] != tag) return;
	right[ord[split_axis[s] * n + p]] = p >= split_pos[s] ? 1u : 0u;   // the first pos - start spheres of the chosen axis' order go left
}
__global__ void __launch_bounds__(kBlock) k_sweep3_flags(const uint32_t* __restrict__ ord, const uint32_t n, const uint32_t* __restrict__ start_of, const uint32_t* __restrict__ split_tag, const uint32_t tag,
                                                         const uint32_t* __restrict__ right, uint32_t* __restrict__ goes_left /*[3n]*/) {
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= 3u * n) return;
	const uint32_t p = t % n;
	goes_left[t] = (split_tag[start_of[p]] == tag && right[ord[t]] == 0u) ? 1u : 0u;
}
__global__ void __launch_bounds__(kBlock) k_sweep3_scatter(const uint32_t* __restrict__ ord, const uint32_t n, const uint32_t* __restrict__ start_of, const uint32_t* __restrict__ split_tag, const uint32_t* __restrict__ split_pos,
                                                           const uint32_t tag, const uint32_t* __restrict__ right, const uint32_t* __restrict__ left_before /*[3n]: exclusive sum of goes_left*/, uint32_t* __restrict__ ord_out) {
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= 3u * n) return;
	const uint32_t axis_base = (t / n) * n, p = t - axis_base, id = ord[t], s = start_of[p];
	uint32_t dest = p;
	if (split_tag[s] == tag) {
		const uint32_t k = left_before[t] - left_before[axis_base + s];   // entries of this run in front of p that go left
		dest = right[id] == 0u ? s + k : split_pos[s] + (p - s - k);
	}
	ord_out[axis_base + dest] = id;
}
// Sum of the inner-slot half areas (the quantity a refit is judged by: cost now / cost when the tree was built).
__global__ void __launch_bounds__(kBlock) k_tree_cost(const float4* __restrict__ wide, const uint32_t n_nodes, double* __restrict__ out) {
	double sum = 0.0;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_nodes * 4u; i += gridDim.x * blockDim.x) {
		const float4 a = wide[static_cast<size_t>(i) * 2u], b = wide[static_cast<size_t>(i) * 2u + 1u];
		if (static_cast<int32_t>(bits(b.z)) >= 0) sum += static_cast<double>(slot_half_area(a, b));
	}
	for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
	if ((threadIdx.x & 31u) == 0u && sum != 0.0) atomicAdd(out, sum);
}

// ---------------------------------------------------------------------------------------------- taps
template <bool LENS>
__global__ void k_tap_generate(const Params p, const uint32_t acc, const LensParams lens, float* __restrict__ out) {
	for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < p.frame.npix; t += gridDim.x * blockDim.x) {
		const PathState s = primary_path<LENS>(p.frame, p.frame.cam, acc, 0u, t, lens);
		float* o = out + static_cast<size_t>(t) * 6u;
		o[0] = s.ox; o[1] = s.oy; o[2] = s.oz; o[3] = s.dx; o[4] = s.dy; o[5] = s.dz;
	}
}
// Traverse / Traverse_shadow on caller-supplied rays (Application.cpp:282-298)
__global__ void k_tap_trace(const SceneDev sc, const float* __restrict__ rays, const float* __restrict__ tfar_in, const uint32_t n,
                            const int use_bvh, const int shadow, float* __restrict__ tfar_out, int32_t* __restrict__ prim_out, uint8_t* __restrict__ occ_out) {
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const float* rr = rays + static_cast<size_t>(i) * 6u;
		const Ray r{rr[0], rr[1], rr[2], rr[3], rr[4], rr[5]};
		uint32_t cs = 0, cb = 0;
		if (!shadow) {
			float best = FLT_MAX; int32_t prim = -1;
			if (use_bvh) traverse_closest<false>(sc.wide, sc.stack_tn_bits, r, &best, &prim, &cs, &cb);
			else for (uint32_t j = 0; j < sc.n_prims; j++) {
				const float4 sp = ldg4(sc.prims + j); float d;
				if (sphere_hit_closest(sp.x, sp.y, sp.z, sp.w, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, &d) && d < best) { best = d; prim = static_cast<int32_t>(j); }
			}
			tfar_out[i] = best; prim_out[i] = prim;
		} else {
			bool occ = false;
			if (use_bvh) occ = traverse_any<false>(sc.wide, r, tfar_in[i], &cs, &cb, sc.parent, 0u);
			else for (uint32_t j = 0; j < sc.n_prims && !occ; j++) {
				const float4 sp = ldg4(sc.prims + j);
				occ = sphere_hit_any(sp.x, sp.y, sp.z, sp.w, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, tfar_in[i]);
			}
			occ_out[i] = occ ? 1 : 0;
		}
	}
}

}  // namespace b2r
