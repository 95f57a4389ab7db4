// b2r.cu — context management and the C ABI of libb2r.so (include/b2r.h). Host code drives the sm_100a kernels of
// b2r_device.cuh; there is no CPU rendering path in this library.
#include "b2r_device.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

using namespace b2r;

namespace {

thread_local std::string g_error;
int fail(int code, const std::string& what) { g_error = what; return code; }
constexpr const char* kDielInvalid = "B2R_FLAG_DIELECTRIC: a material has a non-finite transmission, or is dielectric (max(transmission) > 0) with a transmission outside [0, 1] or 1 + IOR_minus_one not finite or < 1";
#define CU(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return fail(B2R_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); } while (0)

enum KernelKind { KK_GENERATE = 0, KK_BRUTE, KK_CLOSEST, KK_SHADE, KK_SHADOW, KK_ACCUMULATE, KK_RESOLVE, KK_COUNT };

constexpr uint32_t kMaxLanes = 4;
struct BatchArgs {
	uint32_t n; uint32_t acc[kMaxSlots]; unsigned long long fold = ~0ull; CameraParams cam; LensParams lens{0.0f, 0.0f};
	// lanes (run_batch): lane j holds n_lane[j] consecutive samples of the batch in slots [j * lane_slots, j * lane_slots + n_lane[j]); the slots
	// between the lanes hold nothing. lanes == 0: one lane, slots 0..n-1.
	uint32_t lanes = 0, lane_slots = 0, n_lane[kMaxLanes] = {0, 0, 0, 0};
	uint32_t slot_of(uint32_t i) const {  // slot of the i-th sample of the batch
		if (lanes == 0u) return i;
		uint32_t j = 0; while (j + 1u < lanes && i >= n_lane[j]) { i -= n_lane[j]; j++; }
		return j * lane_slots + i;
	}
};
// dst[0] describes the whole batch (k_accumulate), dst[1 + j] lane j's part of it (slot numbers local to the lane)
__global__ void k_set_batch(BatchDev* dst, const BatchArgs a) {
	if (threadIdx.x == 0) { dst[0].n_slots = a.n; dst[0].fold = a.fold; dst[0].cam = a.cam; dst[0].lens = a.lens; }
	if (threadIdx.x < a.n) dst[0].acc[threadIdx.x] = a.acc[threadIdx.x];
	for (uint32_t j = 0; j < kMaxLanes; j++) {
		const uint32_t nj = j < a.lanes ? a.n_lane[j] : 0u;
		if (threadIdx.x == 0) { dst[1 + j].n_slots = nj; dst[1 + j].fold = 0ull; dst[1 + j].cam = a.cam; dst[1 + j].lens = a.lens; }
		if (threadIdx.x < nj) dst[1 + j].acc[threadIdx.x] = a.acc[j * a.lane_slots + threadIdx.x];
	}
}

template <typename T> int dev_alloc(T** p, size_t count) {
	if (*p) { cudaFree(*p); *p = nullptr; }
	if (count == 0) count = 1;
	CU(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
	return B2R_OK;
}
// grow-only variant for the scene tables: a re-upload of a scene of the same size (Application.cpp:508-510 does one per
// geometry edit) reuses the allocations instead of paying cudaFree/cudaMalloc every time
template <typename T> int dev_reserve(T** p, size_t* capacity, size_t count) {
	if (count == 0) count = 1;
	if (*p && *capacity >= count) return B2R_OK;
	if (*p) { cudaFree(*p); *p = nullptr; *capacity = 0; }
	CU(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
	*capacity = count;
	return B2R_OK;
}
template <typename T> void dev_free(T** p) { if (*p) { cudaFree(*p); *p = nullptr; } }

// The scene's device tables: X(element type, name, the length it follows). pack_scene fills the first group (PackedScene uses the same
// names); the tree builds and k_link_tables write wide, parent and leaf_node on the device; hdri is the sky. Every operation on all tables
// (reserve, free, the side copies, binding into Params) walks this list, so a new table is added here and where it is filled and read.
#define B2R_PACKED_TABLES(X) X(float4, prims, LEN_PRIMS) X(int32_t, prim_mat, LEN_PRIMS) X(float4, mat_albedo, LEN_MAT) X(float4, mat_emission, LEN_MAT) \
                             X(float4, mat_f0, LEN_MAT) X(float4, mat_diel, LEN_MAT) X(float4, light_sphere, LEN_LIGHTS) X(float4, light_emit, LEN_LIGHTS)
#define B2R_SCENE_TABLES(X) B2R_PACKED_TABLES(X) X(WideNode, wide, LEN_WIDE) X(uint32_t, parent, LEN_WIDE) X(uint32_t, leaf_node, LEN_PRIMS) X(float4, hdri, LEN_TEXELS) \
                            X(float, sky_marg, LEN_SKY_MARG) X(float, sky_cond, LEN_SKY_COND) X(float, sky_pdf, LEN_SKY_PDF) \
                            X(float4, ltree_nodes, LEN_LTREE_NODES) X(int4, ltree_light, LEN_LTREE_LIGHTS) X(int32_t, ltree_prim_light, LEN_LTREE_PRIMS)
// 0 lights: one (zero) light row. LEN_SKY_*: the sky's tables (B2R_FLAG_SKY_LIGHT), LEN_LTREE_*: the light tree's (B2R_FLAG_LIGHT_TREE), 0 while
// they are not built
enum TableLen { LEN_PRIMS = 0, LEN_MAT, LEN_LIGHTS, LEN_WIDE, LEN_TEXELS, LEN_SKY_MARG, LEN_SKY_COND, LEN_SKY_PDF, LEN_LTREE_NODES, LEN_LTREE_LIGHTS, LEN_LTREE_PRIMS,
                LEN_COUNT };
struct SceneTables {
	template <typename T> struct Table { T* p = nullptr; size_t cap = 0; };
#define X(T, name, len) Table<T> name;
	B2R_SCENE_TABLES(X)
#undef X
	// f(length, the table of each set) for every table in list order, up to the first non-zero return
	template <typename F, typename... S> static int for_each(F&& f, S&... sets) {
		int rc = B2R_OK;
#define X(T, name, len) if (rc == B2R_OK) rc = f(len, sets.name...);
		B2R_SCENE_TABLES(X)
#undef X
		return rc;
	}
};
void free_tables(SceneTables& t) { SceneTables::for_each([](int, auto& x) -> int { dev_free(&x.p); x.cap = 0; return B2R_OK; }, t); }
// The kernels read the tables through Params; `sky` = false leaves hdri null (a scene without ambient light).
void bind_tables(Params& p, const SceneTables& t, bool sky) {
	SceneDev& s = p.scene;
	s.prims = t.prims.p; s.prim_mat = t.prim_mat.p; s.mat_albedo = t.mat_albedo.p; s.mat_emission = t.mat_emission.p; s.mat_f0 = t.mat_f0.p;
	s.light_sphere = t.light_sphere.p; s.light_emit = t.light_emit.p; s.wide = t.wide.p; s.parent = t.parent.p; s.leaf_node = t.leaf_node.p;
	s.hdri = sky ? t.hdri.p : nullptr;
	p.mat_diel = t.mat_diel.p;
	p.sky.marg = t.sky_marg.p; p.sky.cond = t.sky_cond.p; p.sky.pdf = t.sky_pdf.p;
	p.ltree.nodes = t.ltree_nodes.p; p.ltree.light = t.ltree_light.p; p.ltree.prim_light = t.ltree_prim_light.p;
}

// One launch of a batch's rounds: the kernel instantiation, its block size and its grid (kernels_of).
template <typename F> struct Role { F fn = nullptr; int block = 0, grid = 0; };
using BounceKernel = void (*)(const Params, const uint32_t);
struct KernelSet { Role<BounceKernel> brute_first, brute, brute_finish, packet, closest, shade, shadow; Role<void (*)(const Params)> generate; };
// The bits of the key that selects a KernelSet (kernels_of).
enum : uint32_t { KEY_COUNT = 1, KEY_EXACT = 2, KEY_GGX = 4, KEY_LENS = 8, KEY_DIEL = 16, KEY_TN16 = 32, KEY_SKY = 64, KEY_LTREE = 128, KEYS = 256 };

// A stream the batches are traced on (the caller's, or a side's) and what a batch's lanes add to it: lane j > 0 runs on lane_stream[j],
// forked from the stream by ev_fork and joined back by ev_join[j]; one captured graph per lane count (index = lanes).
struct Track {
	cudaStream_t lane_stream[kMaxLanes] = {}; cudaEvent_t ev_fork = nullptr, ev_join[kMaxLanes] = {};
	cudaGraphExec_t exec[kMaxLanes + 1] = {}; bool valid[kMaxLanes + 1] = {};
	uint64_t launches[kMaxLanes + 1] = {};  // kernels one replay of each graph launches (counted while capturing)
	void invalidate() { for (bool& v : valid) v = false; }
	void drop_graphs() { for (cudaGraphExec_t& e : exec) if (e) { cudaGraphExecDestroy(e); e = nullptr; } invalidate(); }  // (nothing of them may still run)
	void destroy() {
		drop_graphs();
		for (uint32_t j = 1; j < kMaxLanes; j++) if (lane_stream[j]) { cudaStreamDestroy(lane_stream[j]); cudaEventDestroy(ev_join[j]); }
		if (ev_fork) cudaEventDestroy(ev_fork);
	}
};

}  // namespace

struct b2r_ctx {
	b2r_config cfg{};
	cudaStream_t stream = nullptr, own_stream = nullptr;
	// scene upload staging: one page-locked block reused by every b2r_upload_scene (no stream synchronisation on the upload path)
	unsigned char* h_stage = nullptr; size_t stage_bytes = 0; cudaEvent_t ev_stage = nullptr; bool stage_busy = false;
	cudaStream_t copy_stream = nullptr; cudaEvent_t ev_resolved = nullptr, ev_copied = nullptr; bool copy_pending = false;  // b2r_resolve_async
	bool have_scene = false, have_camera = false, use_bvh = false;
	uint32_t accumulations = 0;
	uint32_t slots = 8;
	int sm_count = 0;
	// scene
	SceneTables tables;  // the primary tables, written by the scene writes (grow-only: reserve_tables)
	bool scene_diel_valid = true;  // the current scene's materials pass dielectric_materials_valid (checked when B2R_FLAG_DIELECTRIC is turned on)
	// B2R_FLAG_SKY_LIGHT: whether the current sky's texels were checked (sky_texels_valid: only under the flag, or when it is turned on), passed,
	// and are not zero everywhere; whether the sky's tables in `tables` are built for the current sky; the build's scratch
	bool sky_checked = false, sky_valid = true, sky_nonzero = false, sky_built = false; double* d_sky_tmp = nullptr; size_t cap_sky_tmp = 0;
	// B2R_FLAG_LIGHT_TREE: the current light list (geometry[light_geom_idx[i]] and its mean emission, kept so that b2r_set_flags can build the
	// tree later), whether it follows the input rule (light_list_valid), and whether the tree's tables in `tables` are built for the current scene
	std::vector<b2r_sphere> lt_lights; std::vector<float> lt_lum; bool lt_valid = true, lt_built = false; uint32_t lt_nodes = 0;
	WideBvh wide_host; uint64_t wide_key = 0; std::vector<unsigned char> wide_blob; bool have_wide = false;
	uint32_t n_wide = 0;  // wide nodes of the current tree
	// B2R_FLAG_GPU_TREE: the tree was built on the device (no host copy of its nodes); sort scratch; the arrays a later refit needs to match
	bool gpu_tree = false; uint32_t *d_mkey[2] = {nullptr, nullptr}, *d_midx[2] = {nullptr, nullptr}; size_t cap_mkey = 0; uint8_t* d_sort_tmp = nullptr; size_t cap_sort_tmp = 0; uint8_t* d_sweep = nullptr; size_t cap_sweep = 0;  // d_sweep: scratch of the sweep build (B2R_FLAG_GPU_SAH)
	std::vector<b2r_sphere> lazy_prims, lazy_geom; double* d_cost_base = nullptr;
	std::vector<uint32_t> cur_geom_of_prim;  // after a refit into a new BVH order: that order's index -> geometry index (empty: wide_host's)
	uint32_t* d_remap = nullptr; size_t cap_remap = 0;
	uint8_t* d_trace = nullptr; size_t cap_trace = 0;  // b2r_trace_* staging (rays in, results out)
	uint8_t* d_tap = nullptr; size_t cap_tap = 0;      // b2r_trace_kernel: the queue planes, counters and batch descriptor of its launches
	bool wide_refit = false; double* d_cost = nullptr;  // b2r_refit_scene: the device tree no longer equals wide_host
	// where ray origins may lie (leaf_half_extent, b2r_shade.h): bounds of the current spheres + camera + caller-supplied ray origins
	OriginBox obox{}; bool obox_valid = false; float sph_lo[3] = {0, 0, 0}, sph_hi[3] = {0, 0, 0}; float cam_pos[3] = {0, 0, 0};
	LensParams lens{0.0f, 0.0f};  // b2r_set_lens: radius 0 = pinhole (the instantiations without LENS)
	// frame
	float4 *d_A[2] = {nullptr, nullptr}, *d_B[2] = {nullptr, nullptr}, *d_SA = nullptr, *d_SB = nullptr, *d_fb = nullptr;
	float *d_T[2] = {nullptr, nullptr}, *d_SL = nullptr, *d_rad = nullptr, *d_acc = nullptr;
	uint32_t* d_N[2] = {nullptr, nullptr};  // start nodes of the paths' closest-hit walks (QueueDev::N)
	uint8_t *d_ex_slot[2] = {nullptr, nullptr}, *d_ex_key = nullptr; uint16_t* d_ex_act[2] = {nullptr, nullptr}; uint32_t* d_ex_next = nullptr;  // B2R_FLAG_REFERENCE_EXACT
	float2* d_H = nullptr; uint32_t* d_SS = nullptr;
	uint32_t* d_counts = nullptr; size_t counts_bytes = 0;
	unsigned long long* d_stats = nullptr;
	BatchDev* d_batch = nullptr;
	Params params{};
	// launch
	KernelSet kernels[KEYS];  // the kernel set of every key this context has used, with its grids (kernels_of)
	int grid_stream = 0; bool packet_primary = true;
	// twin lanes: a batch of two or more samples is traced as two independent half batches on two streams (own queues, counters and batch
	// descriptors) inside one graph, so that the drained end of every launch of one half is filled by the other half's kernels
	Track main;  // the batches traced on the caller's stream (sides off)
	bool idle = true;  // nothing of this context is running on the device (set by sync_main, cleared by run_batch)
	uint32_t lanes_max = 2; bool lanes_forced = false;  // B2R_LANES given: no per-batch choice
	float lane_grid_frac = 1.0f;
	// sides: consecutive batches alternate between two halves of the queue memory and are TRACED on two library-owned streams, so that the thin
	// late bounces of one batch (and its fold and the frame's resolve) run under the first, fat bounces of the next; only k_accumulate stays on
	// the caller's stream, behind an event, so buckets are still folded in sample order and everything the caller enqueues later (reset,
	// resolve, a scene upload) is ordered behind all tracing enqueued so far
	struct Side {
		cudaStream_t stream = nullptr; Track track;
		cudaEvent_t ev_traced = nullptr, ev_folded = nullptr, ev_sync = nullptr;
		bool folded_valid = false; uint64_t epoch = ~0ull;
		// the side's own copy of the scene arrays (refreshed from the primary ones, device to device, on the side's stream when scene_version has
		// moved on): tracing never reads the primary arrays, so a scene upload does not have to wait for the batch in flight
		SceneTables tables;  // (allocated at the primary tables' capacities)
		bool have_copy = false, refreshed_valid = false; uint64_t scene_version = ~0ull; cudaEvent_t ev_refreshed = nullptr;
	} side[2];
	uint32_t sides = 2, next_side = 0, last_side = 0, spec_side = 0, counts_first = 0;  // counts_first: first counter block of the last batch
	uint64_t scene_epoch = 0;  // bumped by what the side streams must not run ahead of on the caller's stream (counter resets)
	// scene writes (upload, refit, origin-box refit, device tree build): on the caller's stream, or — when the scene is traced through the sides —
	// on the library's upload stream, so that frame N+1's scene copies run while frame N is still tracing from the sides' own copies
	cudaStream_t up_stream = nullptr, scene_st = nullptr; cudaEvent_t ev_uploaded = nullptr, ev_main_mark = nullptr; bool uploaded_valid = false;
	uint64_t scene_version = 0;     // bumped by every scene write
	bool main_reads_scene = false;  // work that reads the primary scene arrays has been enqueued on the caller's stream since the last scene write
	size_t hdri_texels = 0;         // texels of the current sky (side copies)
	uint64_t launches = 0;
	// profiling (B2R_FLAG_NO_GRAPH): events around every launch
	struct Timed { int kind; cudaEvent_t a, b; };
	std::vector<Timed> timed;
	double kernel_ms[8] = {0}; uint64_t kernel_launches[8] = {0};
	// peers' bucket arrays mapped through CUDA IPC (multi-GPU fused resolve)
	std::vector<void*> peer_acc; uint32_t my_rank = 0;
	// team mode (b2r_team_*): peers' bucket arrays, rank 0's framebuffer and every rank's TeamSync block, mapped through CUDA IPC
	// samples traced ahead of the caller: an application that calls Accumulate() once per frame (Application.cpp:379) gets wavefront
	// batches of 2, 4, ... kSpecMax samples as long as nothing invalidates them; the extra samples wait in RAD and are folded by later calls
	uint32_t spec_width = 1, spec_first = 0, spec_count = 0, spec_used = 0; BatchArgs spec_args;  // (spec_args in the slot layout run_batch gave it)
	TeamSync* d_team = nullptr; std::vector<void*> team_acc, team_sync; void* team_fb0 = nullptr; uint32_t team_rank = 0, team_frame = 0; bool team_wait_done = false;
};

namespace {

int ensure_device(b2r_ctx* c) { CU(cudaSetDevice(c->cfg.device)); return B2R_OK; }
// every wait for the caller's stream goes through here: afterwards the device is idle (all tracing enqueued so far precedes that stream's
// position), which run_batch takes into account when it shapes the next batch
cudaError_t sync_main(b2r_ctx* c) { c->idle = true; return cudaStreamSynchronize(c->stream); }
constexpr uint32_t kSpecMax = 16;
constexpr uint32_t kFinishBelow = 12000000u;  // paths entering a bounce below which k_brute_finish takes the rest of a brute-force batch. Measured on C2 (134 M paths
                                              // per batch): 13.72 ms per frame without it, 13.41 at 8 M, 13.34 at 12-16 M, 13.48 at 25 M; B2R_FINISH_BELOW overrides (0 = off)
void drop_speculation(b2r_ctx* c) { c->spec_count = 0; c->spec_used = 0; c->spec_width = 1; }  // scene, camera, sample index or buckets changed under the samples traced ahead

void drop_graph(b2r_ctx* c) {
	drop_speculation(c);  // everything that invalidates the captured graph (camera, scene pointers, flags, frame size) invalidates them too
	if (c->stream) sync_main(c);  // (a launch of a graph may still be running)
	c->main.drop_graphs();
	for (auto& S : c->side) {
		if (S.stream) cudaStreamSynchronize(S.stream);
		S.track.drop_graphs();
	}
}

int alloc_frame(b2r_ctx* c) {
	const uint32_t w = c->cfg.width, h = c->cfg.height, npix = w * h, mb = c->cfg.max_bounces, K = c->cfg.buckets;
	if (c->cfg.samples_in_flight == 0) {  // default: about 128M paths per wavefront batch (keeps the late, thin bounces a small share)
		uint32_t s = (128u << 20) / npix; c->slots = s < 4u ? 4u : s > static_cast<uint32_t>(kMaxSlots) ? static_cast<uint32_t>(kMaxSlots) : s;
	}
	const size_t cap = static_cast<size_t>(c->slots) * npix;
	if (3 * cap >= (1ull << 32)) return fail(B2R_ERR_ARG, "samples_in_flight * pixels too large: the three-plane queue arrays are indexed with 32 bits");
	int rc;
	for (int s = 0; s < 2; s++) {
		if ((rc = dev_alloc(&c->d_A[s], cap))) return rc;
		if ((rc = dev_alloc(&c->d_B[s], cap))) return rc;
		if ((rc = dev_alloc(&c->d_T[s], 3 * cap))) return rc;
		if ((rc = dev_alloc(&c->d_N[s], cap))) return rc;
	}
	if ((rc = dev_alloc(&c->d_H, cap))) return rc;
	if ((rc = dev_alloc(&c->d_SA, cap))) return rc;
	if ((rc = dev_alloc(&c->d_SB, cap))) return rc;
	if ((rc = dev_alloc(&c->d_SL, 3 * cap))) return rc;
	if ((rc = dev_alloc(&c->d_SS, cap))) return rc;
	if ((rc = dev_alloc(&c->d_rad, 3 * cap))) return rc;
	if ((rc = dev_alloc(&c->d_acc, static_cast<size_t>(K) * 3 * npix))) return rc;
	if ((rc = dev_alloc(&c->d_fb, static_cast<size_t>(npix)))) return rc;
	c->counts_bytes = (static_cast<size_t>(mb) + 1) * 4 * sizeof(uint32_t);
	if ((rc = dev_alloc(&c->d_counts, (static_cast<size_t>(mb) + 1) * 4 * kMaxLanes * 2))) return rc;  // one block per lane and side
	CU(cudaMemset(c->d_counts, 0, 2 * kMaxLanes * c->counts_bytes));
	if (!c->d_stats) { if ((rc = dev_alloc(&c->d_stats, static_cast<size_t>(ST_COUNT)))) return rc; CU(cudaMemset(c->d_stats, 0, ST_COUNT * sizeof(unsigned long long))); }
	if (!c->d_batch) { if ((rc = dev_alloc(&c->d_batch, static_cast<size_t>(2 * (1 + kMaxLanes))))) return rc; }  // per side: whole batch + one per lane
	if (c->cfg.flags & B2R_FLAG_REFERENCE_EXACT) {
		for (int s = 0; s < 2; s++) { if ((rc = dev_alloc(&c->d_ex_slot[s], cap))) return rc; if ((rc = dev_alloc(&c->d_ex_act[s], cap / 256))) return rc; }
		if ((rc = dev_alloc(&c->d_ex_key, cap))) return rc;
		if ((rc = dev_alloc(&c->d_ex_next, cap))) return rc;
		CU(cudaMemset(c->d_ex_key, 0, cap));
	}
	CU(cudaMemset(c->d_rad, 0, 3 * cap * sizeof(float)));
	CU(cudaMemset(c->d_acc, 0, static_cast<size_t>(K) * 3 * npix * sizeof(float)));
	Params& p = c->params;
	p.frame.width = w; p.frame.height = h; p.frame.h_tiles = w / 16; p.frame.npix = npix;
	p.frame.h_tiles_magic = magic_for(w / 16); p.frame.npix_magic = magic_for(npix);
	p.frame.max_bounces = mb; p.frame.buckets = K; p.frame.flags = c->cfg.flags;
	{  // k_brute_finish hand-over (brute-force pipeline): default threshold, overridable for measurements
		const char* e = std::getenv("B2R_FINISH_BELOW"); const char* f = std::getenv("B2R_FINISH_FIRST");
		p.frame.finish_below = e ? static_cast<uint32_t>(std::strtoul(e, nullptr, 10)) : kFinishBelow;
		p.frame.finish_first = f ? static_cast<uint32_t>(std::strtoul(f, nullptr, 10)) : 2u;
	}
	for (int s = 0; s < 2; s++) { p.q.A[s] = c->d_A[s]; p.q.B[s] = c->d_B[s]; p.q.T[s] = c->d_T[s]; p.q.N[s] = c->d_N[s]; }
	p.q.H = c->d_H; p.q.SA = c->d_SA; p.q.SB = c->d_SB; p.q.SL = c->d_SL; p.q.SS = c->d_SS; p.q.cap = static_cast<uint32_t>(cap);
	p.cnt.paths = c->d_counts; p.cnt.shadow = c->d_counts + (mb + 1); p.cnt.work_a = c->d_counts + 2 * (mb + 1); p.cnt.work_b = c->d_counts + 3 * (mb + 1);
	p.cnt.stats = c->d_stats;
	p.batch = c->d_batch; p.rad = c->d_rad; p.acc = c->d_acc;
	for (int s = 0; s < 2; s++) { p.ex.slot[s] = c->d_ex_slot[s]; p.ex.act[s] = c->d_ex_act[s]; }
	p.ex.key = c->d_ex_key; p.ex.next_idx = c->d_ex_next;
	c->accumulations = 0;
	drop_graph(c);
	return B2R_OK;
}

// One launch; in profiling mode bracketed by events.
template <typename F> int launch(b2r_ctx* c, int kind, bool profile, F&& f) {
	b2r_ctx::Timed t{kind, nullptr, nullptr};
	if (profile) { CU(cudaEventCreate(&t.a)); CU(cudaEventCreate(&t.b)); CU(cudaEventRecord(t.a, c->stream)); }
	f();
	CU(cudaGetLastError());
	if (profile) { CU(cudaEventRecord(t.b, c->stream)); c->timed.push_back(t); }
	c->launches++;
	return B2R_OK;
}

// The kernel variant (template instantiation of b2r_device.cuh) of every role for one key. The sphere-test counters (COUNT) are built into
// the traversal kernels always, and into the shading kernels only without GGX and without DIELECTRIC. A lens changes bounce 0 only (later
// bounces read their origins from the path records). TN16: stack entries split 16/16 (up to 65536 wide nodes: C3) get immediate shifts;
// other trees read the split from the scene.
template <uint32_t KEY> KernelSet kernel_set() {
	constexpr bool COUNT = KEY & KEY_COUNT, EXACT = KEY & KEY_EXACT, GGX = KEY & KEY_GGX, LENS = KEY & KEY_LENS, DIEL = KEY & KEY_DIEL, TN16 = KEY & KEY_TN16,
	               SKY = KEY & KEY_SKY, LTREE = KEY & KEY_LTREE;
	if constexpr ((EXACT && (GGX || LENS || DIEL)) || (SKY && (EXACT || GGX)) || (LTREE && EXACT)) return {};  // refused by b2r_create, b2r_set_flags and b2r_set_lens: nothing instantiated
	else {
		constexpr bool SHADE_COUNT = COUNT && !GGX && !DIEL && !SKY && !LTREE;
		KernelSet k;
		k.brute_first = {k_bounce_brute<true, SHADE_COUNT, EXACT, GGX, LENS, DIEL, SKY, LTREE>, kBruteBlock};
		k.brute = {k_bounce_brute<false, SHADE_COUNT, EXACT, GGX, false, DIEL, SKY, LTREE>, kBruteBlock};
		k.brute_finish = {k_brute_finish<SHADE_COUNT, GGX, DIEL, SKY, LTREE>, kBruteBlock};
		k.packet = {k_intersect_packet<COUNT, LENS ? B2R_PACKET_RPL_LENS : B2R_PACKET_RPL, LENS>, kTravBlock};
		k.closest = {k_intersect_closest<COUNT, EXACT, TN16 ? 16u : 0u>, kTravBlock};
		k.shade = {k_shade<EXACT, GGX, DIEL, SKY, LTREE>, kBruteBlock};
		k.shadow = {k_intersect_shadow<COUNT>, kTravBlock};
		k.generate = {k_generate<LENS>, kBlock};
		return k;
	}
}
template <uint32_t... KEY> KernelSet kernel_set(uint32_t key, std::integer_sequence<uint32_t, KEY...>) {
	static const KernelSet sets[] = {kernel_set<KEY>()...};
	return sets[key];
}
// The kernel set of the context's flags, lens and tree. Every role's grid is SM count x the resident CTAs of its instantiation at its block
// size, queried once per context and key: run_batch and b2r_trace_kernel look the set up before they enqueue (no query inside a capture).
int kernels_of(b2r_ctx* c, const KernelSet** out) {
	const uint32_t f = c->cfg.flags;
	const bool exact = (f & B2R_FLAG_REFERENCE_EXACT) != 0;
	const uint32_t key = ((f & B2R_FLAG_COUNT_TESTS) ? KEY_COUNT : 0u) | (exact ? KEY_EXACT : 0u) | ((f & B2R_FLAG_GGX) ? KEY_GGX : 0u) |
	                     (c->lens.radius > 0.0f && !exact ? KEY_LENS : 0u) | ((f & B2R_FLAG_DIELECTRIC) ? KEY_DIEL : 0u) | (c->params.scene.stack_tn_bits == 16u ? KEY_TN16 : 0u) |
	                     ((f & B2R_FLAG_SKY_LIGHT) ? KEY_SKY : 0u) | ((f & B2R_FLAG_LIGHT_TREE) ? KEY_LTREE : 0u);
	KernelSet& k = c->kernels[key];
	if (!k.shade.fn) {
		KernelSet s = kernel_set(key, std::make_integer_sequence<uint32_t, KEYS>());
		auto occ = [&](auto& r) -> int {
			int n = 0; CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, reinterpret_cast<const void*>(r.fn), r.block, 0));
			r.grid = (n < 1 ? 1 : n) * c->sm_count; return B2R_OK;
		};
		int rc;
		if ((rc = occ(s.brute_first)) || (rc = occ(s.brute)) || (rc = occ(s.brute_finish)) || (rc = occ(s.packet)) || (rc = occ(s.closest)) || (rc = occ(s.shade)) ||
		    (rc = occ(s.shadow)) || (rc = occ(s.generate))) return rc;
		k = s;
	}
	*out = &k;
	return B2R_OK;
}

// The max_bounces rounds of one batch — or of one lane's half of it — on stream st; p carries that batch's queues, counters and descriptor.
int enqueue_rounds(b2r_ctx* c, const KernelSet& k, const Params& p_in, cudaStream_t st, bool profile, float grid_frac = 1.0f, uint32_t lanes = 1) {
	// (measurement tap, B2R_LANE_GRID: the lanes of a twin batch may be given a fraction of the resident-CTA grid each, so that the two lanes'
	// kernels sit on every SM side by side instead of taking turns)
	auto G = [&](int g) { const int per_sm = g / c->sm_count; int k = static_cast<int>(per_sm * grid_frac + 0.5f); if (k < 1) k = 1; return k * c->sm_count; };
	const bool exact = (c->cfg.flags & B2R_FLAG_REFERENCE_EXACT) != 0;
	if (exact && c->params.scene.n_mat > 64) return fail(B2R_ERR_STATE, "B2R_FLAG_REFERENCE_EXACT: at most 64 materials (RendererPolicy::max_materialID, Renderer.hpp:23)");
	const uint32_t mb = c->cfg.max_bounces;
	Params p = p_in;
	int rc;
	auto run = [&](int kind, const Role<BounceKernel>& r, int grid, uint32_t b) { return launch(c, kind, profile, [&] { r.fn<<<grid, r.block, 0, st>>>(p, b); }); };
	const Role<BounceKernel> rank{k_stream_rank, 256, c->grid_stream};
	if (!c->use_bvh) {
		const bool finish = !exact && p.frame.finish_below != 0u && p.scene.n_prims <= static_cast<uint32_t>(kBruteTile);
		if (!finish) p.frame.finish_below = 0u;  // the hand-over threshold only reaches the kernels when k_brute_finish is launched too
		else if (lanes > 1u) p.frame.finish_below /= lanes;  // the threshold is a batch's; a lane sees 1 / lanes of its paths (C2, two lanes: 13.15 -> 12.80 ms per frame)
		for (uint32_t b = 0; b < mb; b++) {
			// k_brute_finish takes the remaining paths over once few enough are left (a no-op launch otherwise)
			if (finish && b >= p.frame.finish_first && b + 1 < mb && (rc = run(KK_BRUTE, k.brute_finish, k.brute_finish.grid, b))) return rc;
			if ((rc = b == 0 ? run(KK_BRUTE, k.brute_first, k.brute_first.grid, b) : run(KK_BRUTE, k.brute, k.brute.grid, b))) return rc;
			// the reference's stream order for the next bounce (the ranking kernel's time is booked under the brute kind)
			if (exact && b + 1 < mb && (rc = run(KK_BRUTE, rank, rank.grid, b))) return rc;
		}
		return B2R_OK;
	}
	if (!c->packet_primary && (rc = launch(c, KK_GENERATE, profile, [&] { k.generate.fn<<<k.generate.grid, k.generate.block, 0, st>>>(p); }))) return rc;  // (the packet kernel generates the camera rays itself)
	const bool mis = !(c->cfg.flags & B2R_FLAG_NO_MIS);
	for (uint32_t b = 0; b < mb; b++) {
		if (b == 0 && c->packet_primary) { if ((rc = run(KK_CLOSEST, k.packet, G(k.packet.grid), b))) return rc; }  // camera rays: one walk per warp
		else if ((rc = run(KK_CLOSEST, k.closest, G(k.closest.grid), b))) return rc;
		if ((rc = run(KK_SHADE, k.shade, G(k.shade.grid), b))) return rc;
		if (exact && b + 1 < mb && (rc = run(KK_SHADE, rank, rank.grid, b))) return rc;
		if (mis && b + 1 < mb && (rc = run(KK_SHADOW, k.shadow, G(k.shadow.grid), b))) return rc;
	}
	return B2R_OK;
}

// Lane `which` of a batch traced as `lanes` lanes: its own part of every queue array (lane_slots = ceil(slots / lanes) samples' worth, the last
// lane what is left), its own counter block and batch descriptor, and its own part of RAD — lane j's local slot s is slot j * lane_slots + s
// of the whole batch, which is how k_accumulate (whole-batch descriptor) finds it.
// (BVH pipeline only: a side holds half of the samples in flight, and the brute-force pipeline — C2: one 64-sample batch per frame — loses more to
// the smaller batches than the overlap gives back: 13.16 -> 13.09 ms per frame device-resident, but e2e 29.0 -> 28.1 Grays/s)
bool sides_for(const b2r_ctx* c, bool use_bvh) { return c->sides == 2u && use_bvh && !(c->cfg.flags & (B2R_FLAG_NO_GRAPH | B2R_FLAG_REFERENCE_EXACT)) && c->slots >= 2u && c->slots % 2u == 0u; }
bool use_sides(const b2r_ctx* c) { return sides_for(c, c->use_bvh); }
uint32_t batch_cap(const b2r_ctx* c) { return use_sides(c) ? c->slots / 2u : c->slots; }   // samples one batch can hold
uint32_t lane_slots_of(const b2r_ctx* c, uint32_t lanes) { return (batch_cap(c) + lanes - 1u) / lanes; }
// (side = 0 with sides off: the batch owns all the queue memory)
Params lane_params(const b2r_ctx* c, uint32_t which, uint32_t lanes, uint32_t side = 0) {
	Params p = c->params;
	const uint32_t cap_slots = batch_cap(c), ls = lane_slots_of(c, lanes), rel = which * ls, mine = rel >= cap_slots ? 0u : (cap_slots - rel < ls ? cap_slots - rel : ls);
	const size_t npix = p.frame.npix, off = static_cast<size_t>(side * cap_slots + rel) * npix, cap = static_cast<size_t>(mine) * npix;
	for (int s = 0; s < 2; s++) { p.q.A[s] += off; p.q.B[s] += off; p.q.T[s] += 3 * off; p.q.N[s] += off; }
	p.q.H += off; p.q.SA += off; p.q.SB += off; p.q.SL += 3 * off; p.q.SS += off; p.q.cap = static_cast<uint32_t>(cap);
	const uint32_t block = (c->cfg.max_bounces + 1u) * 4u, blk = side * kMaxLanes + which;
	p.cnt.paths += blk * block; p.cnt.shadow += blk * block; p.cnt.work_a += blk * block; p.cnt.work_b += blk * block;
	p.batch = c->d_batch + side * (1u + kMaxLanes) + 1u + which;
	p.rad += 3 * off;
	if (use_sides(c)) bind_tables(p, c->side[side].tables, p.scene.hdri != nullptr);  // a side traces from its own copy of the scene arrays (refresh_side_scene)
	return p;
}
// what k_accumulate sees of a side: that side's whole-batch descriptor and its part of RAD
Params side_params(const b2r_ctx* c, uint32_t side) {
	Params p = c->params;
	p.batch = c->d_batch + side * (1u + kMaxLanes);
	p.rad += 3 * static_cast<size_t>(side * batch_cap(c)) * p.frame.npix;
	return p;
}
// One batch (everything after k_set_batch) on track t, whose own stream st runs lane 0, in side `side`'s part of the queue memory (the
// caller's stream: side 0's): the side's counter blocks reset, then max_bounces rounds per lane, forked from st and joined back before
// anything that follows. fold: the batch's k_accumulate follows on st (which adds in sample order over all lanes).
int enqueue_batch(b2r_ctx* c, const KernelSet& k, Track& t, cudaStream_t st, uint32_t side, uint32_t lanes, bool fold, bool profile) {
	CU(cudaMemsetAsync(c->d_counts + static_cast<size_t>(side) * kMaxLanes * (c->counts_bytes / sizeof(uint32_t)), 0, kMaxLanes * c->counts_bytes, st));
	int rc;
	if (lanes <= 1u) {  // one lane: the whole-batch descriptor is the lane's
		Params p = lane_params(c, 0, 1, side); p.batch = c->d_batch + side * (1u + kMaxLanes);
		if ((rc = enqueue_rounds(c, k, p, st, profile))) return rc;
	} else {
		CU(cudaEventRecord(t.ev_fork, st));
		for (uint32_t j = 1; j < lanes; j++) CU(cudaStreamWaitEvent(t.lane_stream[j], t.ev_fork, 0));
		for (uint32_t j = 0; j < lanes; j++) if ((rc = enqueue_rounds(c, k, lane_params(c, j, lanes, side), j ? t.lane_stream[j] : st, false, c->lane_grid_frac, lanes))) return rc;
		for (uint32_t j = 1; j < lanes; j++) { CU(cudaEventRecord(t.ev_join[j], t.lane_stream[j])); CU(cudaStreamWaitEvent(st, t.ev_join[j], 0)); }
	}
	if (!fold) return B2R_OK;
	return launch(c, KK_ACCUMULATE, profile, [&] { k_accumulate<<<c->grid_stream, kBlock, 0, st>>>(c->params); });
}
// The same batch as a replay of track t's graph for this lane count, captured on first use. An invalidated graph is destroyed once st has
// drained.
int replay_batch(b2r_ctx* c, const KernelSet& k, Track& t, cudaStream_t st, uint32_t side, uint32_t lanes, bool fold) {
	if (!t.valid[lanes]) {
		if (t.exec[lanes]) { CU(st == c->stream ? sync_main(c) : cudaStreamSynchronize(st)); cudaGraphExecDestroy(t.exec[lanes]); t.exec[lanes] = nullptr; }
		if (lanes > 1u && !t.ev_fork) CU(cudaEventCreateWithFlags(&t.ev_fork, cudaEventDisableTiming));
		for (uint32_t j = 1; j < lanes; j++) if (!t.lane_stream[j]) {
			CU(cudaStreamCreateWithFlags(&t.lane_stream[j], cudaStreamNonBlocking)); CU(cudaEventCreateWithFlags(&t.ev_join[j], cudaEventDisableTiming));
		}
		cudaGraph_t graph = nullptr;
		const uint64_t before = c->launches;
		CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
		int rc = enqueue_batch(c, k, t, st, side, lanes, fold, false);
		cudaError_t e = cudaStreamEndCapture(st, &graph);
		t.launches[lanes] = c->launches - before; c->launches = before;
		if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
		if (e != cudaSuccess) return fail(B2R_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
		e = cudaGraphInstantiate(&t.exec[lanes], graph, 0);
		cudaGraphDestroy(graph);
		if (e != cudaSuccess) return fail(B2R_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
		t.valid[lanes] = true;
	}
	CU(cudaGraphLaunch(t.exec[lanes], st));
	c->launches += t.launches[lanes];
	return B2R_OK;
}

int refresh_side_scene(b2r_ctx* c, uint32_t sidx);
// One wavefront batch of args.n samples (args.acc[0..n) in sample order). Two or more samples are traced as lanes: run_batch moves every
// lane's samples to the slots that lane owns and leaves args in that layout (the caller may keep it: samples traced ahead).
int run_batch(b2r_ctx* c, BatchArgs& args) {
	const bool no_graph = (c->cfg.flags & B2R_FLAG_NO_GRAPH) != 0;
	uint32_t lanes = 1;
	if (!no_graph && !(c->cfg.flags & B2R_FLAG_REFERENCE_EXACT)) {
		if (c->lanes_max >= 4u && args.n >= 4u && batch_cap(c) % 4u == 0u) lanes = 4;
		else if (c->lanes_max >= 2u && args.n >= 2u && batch_cap(c) >= 2u) lanes = 2;
		// With sides a batch normally runs under the previous one (the other side's), and then ONE lane of full-size launches is the better
		// shape (C3, frames enqueued back to back: 20.7 ms per frame against 21.4 with two lanes per side). A batch that has nothing to run
		// under — the caller has waited for the device since the last batch, or this side must first wait for a scene upload or refit on the
		// caller's stream — overlaps nothing but itself, and keeps its lanes.
		if (use_sides(c) && !c->lanes_forced && !c->idle && c->side[c->next_side].epoch == c->scene_epoch) lanes = 1;
	}
	c->idle = false;
	if (lanes > 1u) {
		const uint32_t n = args.n, ls = lane_slots_of(c, lanes);
		uint32_t acc[kMaxSlots]; for (uint32_t i = 0; i < n; i++) acc[i] = args.acc[i];
		unsigned long long fold = 0ull; uint32_t i = 0, span = 0;
		for (uint32_t s = 0; s < static_cast<uint32_t>(kMaxSlots); s++) args.acc[s] = 0u;
		for (uint32_t j = 0; j < lanes; j++) {
			const uint32_t nj = n / lanes + (j < n % lanes ? 1u : 0u);   // the first lanes take the remainder: never more than ceil(n / lanes) <= lane_slots
			args.n_lane[j] = nj;
			for (uint32_t k = 0; k < nj; k++, i++) { const uint32_t slot = j * ls + k; args.acc[slot] = acc[i]; if ((args.fold >> i) & 1ull) fold |= 1ull << slot; if (slot + 1u > span) span = slot + 1u; }
		}
		args.lanes = lanes; args.lane_slots = ls; args.n = span; args.fold = fold;
	} else { args.lanes = 0; args.lane_slots = 0; if (args.n < 64u) args.fold &= (1ull << args.n) - 1ull; }
	args.cam = c->params.frame.cam; args.lens = c->lens;  // the camera and lens travel with the batch descriptor: a camera move leaves the captured graph alone
	const KernelSet* k = nullptr;
	{ const int rc = kernels_of(c, &k); if (rc) return rc; }
	if (use_sides(c)) {
		const uint32_t sidx = c->next_side; c->next_side ^= 1u;
		b2r_ctx::Side& S = c->side[sidx];
		if (!S.stream) {
			CU(cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
			for (cudaEvent_t* e : {&S.ev_traced, &S.ev_folded, &S.ev_sync}) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
		}
		// the side must not run ahead of scene copies / refits enqueued on the caller's stream since it last looked, nor overwrite its part of
		// RAD before the previous batch it traced has been folded
		if (S.epoch != c->scene_epoch) { CU(cudaEventRecord(S.ev_sync, c->stream)); CU(cudaStreamWaitEvent(S.stream, S.ev_sync, 0)); S.epoch = c->scene_epoch; }
		if (S.folded_valid) CU(cudaStreamWaitEvent(S.stream, S.ev_folded, 0));
		{ const int rc = refresh_side_scene(c, sidx); if (rc) return rc; }
		k_set_batch<<<1, kMaxSlots, 0, S.stream>>>(c->d_batch + sidx * (1u + kMaxLanes), args);
		CU(cudaGetLastError());
		{ const int rc = replay_batch(c, *k, S.track, S.stream, sidx, lanes, false); if (rc) return rc; }
		CU(cudaEventRecord(S.ev_traced, S.stream));
		// the fold stays on the caller's stream: buckets are added to in sample order, behind whatever the caller enqueued before (reset)
		CU(cudaStreamWaitEvent(c->stream, S.ev_traced, 0));
		k_accumulate<<<c->grid_stream, kBlock, 0, c->stream>>>(side_params(c, sidx));
		CU(cudaGetLastError());
		CU(cudaEventRecord(S.ev_folded, c->stream)); S.folded_valid = true;
		c->launches += 1u;
		c->last_side = sidx; c->counts_first = sidx * kMaxLanes;
		return B2R_OK;
	}
	c->counts_first = 0; c->main_reads_scene = true;  // (this batch traces from the primary scene arrays, on the caller's stream)
	k_set_batch<<<1, kMaxSlots, 0, c->stream>>>(c->d_batch, args);
	CU(cudaGetLastError());
	if (no_graph) return enqueue_batch(c, *k, c->main, c->stream, 0, 1, true, true);
	return replay_batch(c, *k, c->main, c->stream, 0, lanes, true);
}

int collect_timings(b2r_ctx* c) {
	if (c->timed.empty()) return B2R_OK;
	CU(sync_main(c));
	for (auto& t : c->timed) {
		float ms = 0.0f; CU(cudaEventElapsedTime(&ms, t.a, t.b));
		c->kernel_ms[t.kind] += ms; c->kernel_launches[t.kind]++;
		cudaEventDestroy(t.a); cudaEventDestroy(t.b);
	}
	c->timed.clear();
	return B2R_OK;
}

bool owns_sample(const b2r_ctx* c, uint32_t acc) {
	const uint32_t stride = c->cfg.bucket_stride;
	if (stride <= 1) return true;
	return ((acc % c->cfg.buckets) % stride) == c->cfg.bucket_first;
}


// Scene writes. begin: picks the stream (see b2r_ctx::up_stream) and orders it behind whatever still reads the primary arrays — a side's
// device-to-device refresh, or work on the caller's stream. end: the caller's stream is ordered behind the write (nothing it enqueued
// earlier waits), and the sides learn that their copies are stale.
void free_side_scenes(b2r_ctx* c) {
	for (auto& S : c->side) {
		free_tables(S.tables);
		S.have_copy = false; S.scene_version = ~0ull;
		S.track.invalidate();  // the captured graphs hold the old addresses
	}
}
// Grow-only reserve of the primary tables for a scene write, len[] elements each (a length of 0 leaves its tables alone). A table that has
// to grow is replaced while it may be in use: first nothing may be running any more, and the sides' copies go too.
int reserve_tables(b2r_ctx* c, const size_t (&len)[LEN_COUNT]) {
	bool grow = false;
	SceneTables::for_each([&](int l, auto& t) -> int { grow = grow || len[l] > t.cap; return B2R_OK; }, c->tables);
	if (grow) {
		CU(sync_main(c)); if (c->up_stream) CU(cudaStreamSynchronize(c->up_stream));
		for (auto& S : c->side) if (S.stream) CU(cudaStreamSynchronize(S.stream));
		free_side_scenes(c);
	}
	return SceneTables::for_each([&](int l, auto& t) -> int { return len[l] ? dev_reserve(&t.p, &t.cap, len[l]) : B2R_OK; }, c->tables);
}
int begin_scene_write(b2r_ctx* c, bool traced_through_sides) {
	cudaStream_t st = c->stream;
	if (traced_through_sides) {
		if (!c->up_stream) { CU(cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking)); CU(cudaEventCreateWithFlags(&c->ev_main_mark, cudaEventDisableTiming)); }
		st = c->up_stream;
		if (c->main_reads_scene) { CU(cudaEventRecord(c->ev_main_mark, c->stream)); CU(cudaStreamWaitEvent(st, c->ev_main_mark, 0)); c->main_reads_scene = false; }
	}
	for (auto& S : c->side) if (S.refreshed_valid) CU(cudaStreamWaitEvent(st, S.ev_refreshed, 0));
	c->scene_st = st;
	return B2R_OK;
}
int end_scene_write(b2r_ctx* c) {
	if (!c->ev_uploaded) CU(cudaEventCreateWithFlags(&c->ev_uploaded, cudaEventDisableTiming));
	CU(cudaEventRecord(c->ev_uploaded, c->scene_st)); c->uploaded_valid = true;
	if (c->scene_st != c->stream) CU(cudaStreamWaitEvent(c->stream, c->ev_uploaded, 0));
	else c->main_reads_scene = true;  // (written on the caller's stream: the next write on the upload stream has to get behind it)
	c->scene_version++;
	c->scene_st = c->stream;
	return B2R_OK;
}
// A side's copy of the scene, brought up to date on the side's own stream before it traces.
int refresh_side_scene(b2r_ctx* c, uint32_t sidx) {
	b2r_ctx::Side& S = c->side[sidx];
	if (S.have_copy && S.scene_version == c->scene_version) return B2R_OK;
	const SceneDev& sc = c->params.scene;
	if (!S.have_copy) {
		const int rc = SceneTables::for_each([](int, auto& s, const auto& m) -> int { s.cap = m.cap; return dev_alloc(&s.p, m.cap); }, S.tables, c->tables);
		if (rc) return rc;
		if (!S.ev_refreshed) CU(cudaEventCreateWithFlags(&S.ev_refreshed, cudaEventDisableTiming));
		S.have_copy = true;
		S.track.invalidate();
	}
	if (c->uploaded_valid) CU(cudaStreamWaitEvent(S.stream, c->ev_uploaded, 0));
	const size_t len[LEN_COUNT] = {sc.n_prims, sc.n_mat, sc.n_lights ? sc.n_lights : 1u, c->n_wide, sc.hdri ? c->hdri_texels : 0u, c->sky_built ? c->params.sky.rows + 1u : 0u,
	                               c->sky_built ? static_cast<size_t>(c->params.sky.rows) * (c->params.sky.cols + 1u) : 0u, c->sky_built ? c->hdri_texels : 0u,
	                               c->lt_built ? 2u * static_cast<size_t>(c->lt_nodes) : 0u, c->lt_built ? sc.n_lights : 0u, c->lt_built ? sc.n_prims : 0u};
	const int rc = SceneTables::for_each([&](int l, auto& s, const auto& m) -> int {
		const size_t bytes = len[l] * sizeof(*m.p);
		if (bytes) CU(cudaMemcpyAsync(s.p, m.p, bytes, cudaMemcpyDeviceToDevice, S.stream));
		return B2R_OK;
	}, S.tables, c->tables);
	if (rc) return rc;
	CU(cudaEventRecord(S.ev_refreshed, S.stream)); S.refreshed_valid = true; S.scene_version = c->scene_version;
	return B2R_OK;
}

// B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH / B2R_FLAG_GPU_SAH3: links of the sweep tree, written into c->tables.wide level by level (b2r_device.cuh
// k_sweep_*; host twins build_sweep_tree / build_sweep3_tree). `curve_order` = the radix sort's output for the curve sweep (the spheres in
// Hilbert order), null for the three-axis sweep (which sorts the spheres by centre x, y and z itself). One 4-byte read-back per level tells
// the host how many nodes the next level has. *built stays false when the tree would be deeper than kSweepMaxLevels (the caller links the
// packed tree).
int sweep_build(b2r_ctx* c, const uint32_t* curve_order, uint32_t n, bool* built) {
	*built = false;
	const bool three = curve_order == nullptr;
	cudaStream_t st = c->scene_st;
	if (n > 0x3fffffffu) return fail(B2R_ERR_ARG, "sweep build: too many spheres");
	const size_t cap = n / 2u + 1u;  // runs of two or more spheres on one level
	const size_t n3 = three ? 3u * static_cast<size_t>(n) : 0u;
	size_t t_sum = 0, t_sum3 = 0, t_sort = 0;
	CU(cub::DeviceScan::ExclusiveSum(nullptr, t_sum, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), static_cast<int>(cap + 1u), st));
	if (three) {
		CU(cub::DeviceScan::ExclusiveSum(nullptr, t_sum3, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), static_cast<int>(n3), st));
		CU(cub::DeviceRadixSort::SortPairs(nullptr, t_sort, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), static_cast<int>(n), 0, 32, st));
	}
	const size_t t_cub = std::max(t_sum, std::max(t_sum3, t_sort));
	const uint32_t tiles = (n + kSweepTile - 1u) / kSweepTile;
	size_t off = 0; auto take = [&](size_t bytes) { const size_t at = off; off += (bytes + 255u) & ~static_cast<size_t>(255u); return at; };
	const size_t o_box = take(n * sizeof(SweepItem)), o_tiles = take(4u * static_cast<size_t>(tiles) * sizeof(SweepItem)), o_cut = take(n * sizeof(unsigned long long)),
	             o_area = take(n * sizeof(float)), o_head = take(n * sizeof(uint32_t)), o_kids0 = take(cap * sizeof(SweepKids)), o_kids1 = take(cap * sizeof(SweepKids)),
	             o_inner = take((cap + 1u) * sizeof(uint32_t)), o_before = take((cap + 1u) * sizeof(uint32_t)), o_cub = take(t_cub),
	             // three-axis sweep only: keys / orders (ping-pong) / per-position run start / per-run cut notes / per-sphere side / partition counts
	             o_keys = take(n3 * 4u), o_keys2 = take(three ? n * 4u : 0u), o_ord0 = take(n3 * 4u), o_ord1 = take(n3 * 4u), o_start = take(three ? n * 4u : 0u), o_tag = take(three ? n * 4u : 0u),
	             o_spos = take(three ? n * 4u : 0u), o_sax = take(three ? n * 4u : 0u), o_right = take(three ? n * 4u : 0u), o_left = take(n3 * 4u), o_lsum = take(n3 * 4u);
	int rc; if ((rc = dev_reserve(&c->d_sweep, &c->cap_sweep, off))) return rc;
	uint8_t* base = c->d_sweep;
	auto u32 = [&](size_t o) { return reinterpret_cast<uint32_t*>(base + o); };
	SweepItem *box = reinterpret_cast<SweepItem*>(base + o_box), *tile_f = reinterpret_cast<SweepItem*>(base + o_tiles), *tile_b = tile_f + tiles, *carry_f = tile_b + tiles, *carry_b = carry_f + tiles;
	unsigned long long* cut_of = reinterpret_cast<unsigned long long*>(base + o_cut); float* area_of = reinterpret_cast<float*>(base + o_area); uint32_t* head = u32(o_head);
	SweepKids* kids[2] = {reinterpret_cast<SweepKids*>(base + o_kids0), reinterpret_cast<SweepKids*>(base + o_kids1)}; uint32_t *inner = u32(o_inner), *before = u32(o_before);
	uint32_t *keys = u32(o_keys), *keys2 = u32(o_keys2), *ord[2] = {u32(o_ord0), u32(o_ord1)}, *start_of = u32(o_start), *split_tag = u32(o_tag), *split_pos = u32(o_spos), *split_axis = u32(o_sax),
	         *right = u32(o_right), *goes_left = u32(o_left), *left_before = u32(o_lsum);
	void* cub_tmp = base + o_cub;
	auto grid = [](size_t threads) { return static_cast<uint32_t>((threads + kBlock - 1u) / kBlock); };
	int oc = 0;  // which of ord[] holds the current orders
	if (!three) k_sweep_boxes<<<grid(n), kBlock, 0, st>>>(c->tables.prims.p, curve_order, n, box, head, kids[0]);
	else {
		k_sweep3_boxes<<<grid(n), kBlock, 0, st>>>(c->tables.prims.p, n, box, keys, ord[1], head, split_tag, kids[0]);   // ord[1]: 0 .. n-1 three times
		for (uint32_t ax = 0; ax < 3u; ax++) {   // stable: equal coordinates keep the sphere order
			size_t t = t_cub;
			CU(cub::DeviceRadixSort::SortPairs(cub_tmp, t, keys + ax * static_cast<size_t>(n), keys2, ord[1] + ax * static_cast<size_t>(n), ord[0] + ax * static_cast<size_t>(n), static_cast<int>(n), 0, 32, st));
		}
	}
	c->launches++;
	std::vector<uint32_t> lf(1, 0u);
	uint32_t m = 1u, tag = 0u; int cur = 0;
	while (m) {
		if (lf.size() > kSweepMaxLevels) return B2R_OK;
		const uint32_t first = lf.back(), child_first = first + m;
		if (child_first > n) return fail(B2R_ERR_BVH, "sweep build: more nodes than spheres");
		lf.push_back(child_first);
		for (int round = 0; round < 3; round++) {
			if (!three) {
				k_sweep_tiles<<<tiles, kSweepTile, 0, st>>>(box, nullptr, head, n, tile_f, tile_b, cut_of);
				k_sweep_carry<<<2, kSweepTile, 0, st>>>(tile_f, tile_b, tiles, carry_f, carry_b);
				k_sweep_cuts<<<tiles, kSweepTile, 0, st>>>(box, nullptr, head, n, carry_f, carry_b, cut_of, area_of, 0xffffffffu, nullptr);
				k_sweep_open<<<grid(m + 1u), kBlock, 0, st>>>(kids[cur], m, cut_of, area_of, head, round == 2 ? inner : nullptr);
				continue;
			}
			tag++;
			for (uint32_t ax = 0; ax < 3u; ax++) {
				const uint32_t* o = ord[oc] + ax * static_cast<size_t>(n);
				k_sweep_tiles<<<tiles, kSweepTile, 0, st>>>(box, o, head, n, tile_f, tile_b, ax == 0u ? cut_of : nullptr);
				k_sweep_carry<<<2, kSweepTile, 0, st>>>(tile_f, tile_b, tiles, carry_f, carry_b);
				k_sweep_cuts<<<tiles, kSweepTile, 0, st>>>(box, o, head, n, carry_f, carry_b, cut_of, area_of, ax, ax == 0u ? start_of : nullptr);
			}
			k_sweep3_open<<<grid(m + 1u), kBlock, 0, st>>>(kids[cur], m, cut_of, area_of, head, split_tag, split_pos, split_axis, tag, round == 2 ? inner : nullptr);
			k_sweep3_mark<<<grid(n), kBlock, 0, st>>>(ord[oc], n, start_of, split_tag, split_pos, split_axis, tag, right);
			k_sweep3_flags<<<grid(n3), kBlock, 0, st>>>(ord[oc], n, start_of, split_tag, tag, right, goes_left);
			size_t t = t_cub;
			CU(cub::DeviceScan::ExclusiveSum(cub_tmp, t, goes_left, left_before, static_cast<int>(n3), st));
			k_sweep3_scatter<<<grid(n3), kBlock, 0, st>>>(ord[oc], n, start_of, split_tag, split_pos, tag, right, left_before, ord[oc ^ 1]);
			oc ^= 1;
		}
		size_t t = t_cub;
		CU(cub::DeviceScan::ExclusiveSum(cub_tmp, t, inner, before, static_cast<int>(m + 1u), st));
		k_sweep_emit<<<grid(m), kBlock, 0, st>>>(kids[cur], m, before, three ? ord[oc] : curve_order, reinterpret_cast<float4*>(c->tables.wide.p), first, child_first, kids[cur ^ 1]);
		c->launches += three ? 40u : 13u;
		uint32_t total = 0u;
		CU(cudaMemcpyAsync(&total, before + m, sizeof total, cudaMemcpyDeviceToHost, st)); CU(cudaStreamSynchronize(st));
		CU(cudaGetLastError());
		if (total > cap) return fail(B2R_ERR_BVH, "sweep build: inconsistent run count");
		m = total; cur ^= 1;
	}
	WideBvh& w = c->wide_host;
	w.level_first = lf; w.depth = static_cast<uint32_t>(lf.size()) - 1u; w.max_stack = 3u * w.depth;
	c->n_wide = lf.back();
	uint32_t node_bits = 1; while ((1ull << node_bits) < c->n_wide) node_bits++;
	w.tn_bits = 32u - node_bits < 29u ? 32u - node_bits : 29u;
	*built = true;
	return B2R_OK;
}

// Boxes of the device tree for the current origin box: one k_refit_level launch per BFS level, deepest first (stream order is the
// dependency). remap (device, may be null) re-links leaves into a new BVH order.
int launch_refit_levels(b2r_ctx* c, const uint32_t* d_remap) {
	const std::vector<uint32_t>& lf = c->wide_host.level_first;
	for (size_t l = lf.size() - 1; l-- > 0;) {
		const uint32_t first = lf[l], count = lf[l + 1] - lf[l];
		k_refit_level<<<(count * 4u + kBlock - 1u) / kBlock, kBlock, 0, c->scene_st>>>(reinterpret_cast<float4*>(c->tables.wide.p), c->tables.prims.p, d_remap, c->obox, first, count);
		c->launches++;
	}
	CU(cudaGetLastError());
	return B2R_OK;
}
// parent[] / leaf_node[] of the device tree (where k_intersect_shadow starts and how it climbs), read off the tree itself
int launch_link_tables(b2r_ctx* c) {
	k_link_tables<<<(c->n_wide * 4u + kBlock - 1u) / kBlock, kBlock, 0, c->scene_st>>>(reinterpret_cast<const float4*>(c->tables.wide.p), c->n_wide, c->tables.parent.p, c->tables.leaf_node.p);
	CU(cudaGetLastError()); c->launches++;
	return B2R_OK;
}
// The points the camera's rays leave from, for the origin box (out: up to two points, returns how many): none before b2r_set_camera, the
// eye without a lens, and with a lens of radius R the corners pos - R and pos + R of the cube that holds the lens disk in any orientation.
// A lens origin pos + orient * L can round a few ulp beyond that cube; the origin box's slack (origin_box_rule: an eighth of the extent, which
// is at least 2R, plus 1 on every side) absorbs that whenever ulp(|pos| + R) < R / 4 + 1, i.e. unless the eye lies more than ~2^24 lens radii
// (and units) from the origin. DESIGN §2's domain (origins below 2^61) holds for lens origins as for any other.
uint32_t camera_origins(const b2r_ctx* c, float out[6]) {
	if (!c->have_camera) return 0u;
	const float r = c->lens.radius;
	if (r == 0.0f) { for (int k = 0; k < 3; k++) out[k] = c->cam_pos[k]; return 1u; }
	for (int k = 0; k < 3; k++) { out[k] = c->cam_pos[k] - r; out[3 + k] = c->cam_pos[k] + r; }
	return 2u;
}
// Ray origins about to be used (camera position, caller-supplied rays) must lie in the origin box the leaf extents were computed for;
// if they do not, the box grows and the device tree's boxes are recomputed for it (tens of microseconds; the box has an eighth of
// slack on every side, so an interactive camera move does not get here every frame).
int ensure_origin_box(b2r_ctx* c, const float* points, uint32_t n_points) {
	if (c->obox_valid && origin_box_holds(c->obox, points, n_points)) return B2R_OK;
	std::vector<float> extra(points, points + 3 * static_cast<size_t>(n_points));
	float cam[6]; const uint32_t n_cam = camera_origins(c, cam);
	extra.insert(extra.end(), cam, cam + 3 * n_cam);
	if (c->obox_valid) { extra.insert(extra.end(), c->obox.lo, c->obox.lo + 3); extra.insert(extra.end(), c->obox.hi, c->obox.hi + 3); }  // never shrinks between uploads
	c->obox = origin_box_rule(c->sph_lo, c->sph_hi, extra.data(), static_cast<uint32_t>(extra.size() / 3)); c->obox_valid = true;
	if (c->have_wide && !c->gpu_tree) wide_fill_boxes(c->wide_host, c->wide_host.prims.data(), c->obox);  // the host copy (and its reference cost) follows: same routine, same result
	if (c->have_scene && c->have_wide) {
		int rc = begin_scene_write(c, use_sides(c)); if (rc) return rc;
		if ((rc = launch_refit_levels(c, nullptr))) return rc;
		return end_scene_write(c);
	}
	return B2R_OK;
}

// B2R_FLAG_SKY_LIGHT (DESIGN §2): the flags it cannot be combined with (null: none)
const char* sky_flag_conflict(uint32_t flags) {
	if (!(flags & B2R_FLAG_SKY_LIGHT)) return nullptr;
	if (flags & B2R_FLAG_REFERENCE_EXACT) return "B2R_FLAG_SKY_LIGHT cannot be combined with B2R_FLAG_REFERENCE_EXACT";
	if (flags & B2R_FLAG_NO_MIS) return "B2R_FLAG_SKY_LIGHT cannot be combined with B2R_FLAG_NO_MIS (there is no light sampling to add the sky to)";
	if (flags & B2R_FLAG_GGX) return "B2R_FLAG_SKY_LIGHT cannot be combined with B2R_FLAG_GGX (Closure<GGX>::pdf is 0: the sky's MIS weights need the BSDF's pdf)";
	return nullptr;
}
// whether `flags` sample the current sky: a sky (ambient > 0) whose texels are not zero everywhere
bool sky_sampled(const b2r_ctx* c, uint32_t flags) { return (flags & B2R_FLAG_SKY_LIGHT) && c->params.scene.has_ambient && c->sky_nonzero; }
// SkyDev's scalars and LightTreeDev::sel_scale for the context's flags and scene (the tables' pointers are bound with the others)
void set_sky_scalars(b2r_ctx* c) {
	SkyDev& k = c->params.sky; const SceneDev& s = c->params.scene;
	k.p_sky = !sky_sampled(c, c->cfg.flags) ? 0.0f : s.n_lights == 0u ? 1.0f : 0.5f;
	k.light_sel_pdf = s.n_lights ? (1.0f - k.p_sky) / static_cast<float>(s.n_lights) : 0.0f;
	k.cols = s.hdri_w > 1 ? static_cast<uint32_t>(s.hdri_w - 1) : 1u; k.rows = s.hdri_h > 1 ? static_cast<uint32_t>(s.hdri_h - 1) : 1u;
	c->params.ltree.sel_scale = s.n_lights ? 1.0f - k.p_sky : 0.0f;  // (B2R_FLAG_LIGHT_TREE)
}
// lengths of the sky's tables for a w x h texture (reserve_tables)
void sky_table_lens(int32_t w, int32_t h, size_t (&len)[LEN_COUNT]) {
	const size_t cols = w > 1 ? static_cast<size_t>(w - 1) : 1u, rows = h > 1 ? static_cast<size_t>(h - 1) : 1u;
	len[LEN_SKY_MARG] = rows + 1u; len[LEN_SKY_COND] = rows * (cols + 1u); len[LEN_SKY_PDF] = static_cast<size_t>(w) * static_cast<size_t>(h);
}
// The sky's tables from the device copy of the texture, on the scene-write stream (k_sky_*, b2r_device.cuh; tables reserved by the caller)
int launch_sky_build(b2r_ctx* c, int32_t w, int32_t h, const float amb[3]) {
	const uint32_t cols = w > 1 ? static_cast<uint32_t>(w - 1) : 1u, rows = h > 1 ? static_cast<uint32_t>(h - 1) : 1u;
	int rc; if ((rc = dev_reserve(&c->d_sky_tmp, &c->cap_sky_tmp, 2u * static_cast<size_t>(rows) + 1u))) return rc;
	const SkyBuild b{c->tables.hdri.p, w, cols, rows, {amb[0], amb[1], amb[2]}, c->d_sky_tmp, c->d_sky_tmp + rows, c->d_sky_tmp + 2u * rows,
	                 c->tables.sky_marg.p, c->tables.sky_cond.p, c->tables.sky_pdf.p};
	const cudaStream_t st = c->scene_st;
	const uint32_t row_grid = static_cast<uint32_t>((static_cast<size_t>(rows) * 32u + kBlock - 1u) / kBlock);
	const size_t texels = static_cast<size_t>(w) * static_cast<size_t>(h);
	k_sky_rows<<<row_grid, kBlock, 0, st>>>(b);
	k_sky_floor<<<1, 32, 0, st>>>(b);
	k_sky_cond<<<row_grid, kBlock, 0, st>>>(b);
	k_sky_marg<<<1, 32, 0, st>>>(b);
	k_sky_pdf<<<static_cast<uint32_t>((texels + kBlock - 1u) / kBlock), kBlock, 0, st>>>(b, static_cast<uint32_t>(h));
	CU(cudaGetLastError()); c->launches += 5;
	return B2R_OK;
}
constexpr const char* kSkyInvalid = "B2R_FLAG_SKY_LIGHT: a sky texel is not finite, or negative, in a channel whose ambient is > 0";

struct UploadPart { void* dst; const void* src; size_t bytes; };
int stage_upload(b2r_ctx* c, const UploadPart* parts, size_t n_parts);

// B2R_FLAG_LIGHT_TREE (DESIGN §2): the flags it cannot be combined with (null: none)
const char* light_tree_flag_conflict(uint32_t flags) {
	if (!(flags & B2R_FLAG_LIGHT_TREE)) return nullptr;
	if (flags & B2R_FLAG_REFERENCE_EXACT) return "B2R_FLAG_LIGHT_TREE cannot be combined with B2R_FLAG_REFERENCE_EXACT";
	if (flags & B2R_FLAG_NO_MIS) return "B2R_FLAG_LIGHT_TREE cannot be combined with B2R_FLAG_NO_MIS (there is no light sampling to pick lights for)";
	return nullptr;
}
constexpr const char* kLightsInvalid = "B2R_FLAG_LIGHT_TREE: a light index appears twice, two lights are equal spheres, or a light's emission is not finite or is negative";
// The light list of a scene write, kept for a tree build by a later b2r_set_flags: geometry[light_geom_idx[i]] and its material's mean emission
void keep_light_list(b2r_ctx* c, const b2r_material* materials, const int32_t* light_geom_idx, uint32_t n_lights, const b2r_sphere* geometry, bool valid) {
	c->lt_lights.resize(n_lights); c->lt_lum.resize(n_lights); c->lt_valid = valid;
	for (uint32_t i = 0; i < n_lights; i++) {
		c->lt_lights[i] = geometry[light_geom_idx[i]];
		const float* e = materials[c->lt_lights[i].material_ID].emission;
		c->lt_lum[i] = ((e[0] + e[1]) + e[2]) / 3.0f;
	}
}
// The light tree of the kept light list over the BVH-order spheres, and the lengths of its tables (reserve_tables)
void build_kept_light_tree(const b2r_ctx* c, const float4* prims, const int32_t* prim_mat, uint32_t n_prims, LightTree& lt, size_t (&len)[LEN_COUNT]) {
	build_light_tree(c->lt_lights.data(), c->lt_lum.data(), static_cast<uint32_t>(c->lt_lights.size()), prims, prim_mat, n_prims, lt);
	len[LEN_LTREE_NODES] = lt.nodes.size(); len[LEN_LTREE_LIGHTS] = lt.light.size(); len[LEN_LTREE_PRIMS] = lt.prim_light.size();
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

static int team_before_bucket_write(b2r_ctx* c);
const char* b2r_last_error(void) { return g_error.c_str(); }
int b2r_abi_version(void) { return B2R_ABI_VERSION; }

int b2r_create(b2r_ctx** out, const b2r_config* cfg) {
	if (!out || !cfg) return fail(B2R_ERR_ARG, "null argument");
	*out = nullptr;
	if (cfg->width == 0 || cfg->height == 0 || cfg->width % 16 || cfg->height % 16) return fail(B2R_ERR_ARG, "width/height must be non-zero multiples of 16 (Renderer::RequiredTiling)");
	if (static_cast<uint64_t>(cfg->width) * cfg->height > kPixMask) return fail(B2R_ERR_ARG, "image too large (2^26 pixels max)");
	if (cfg->buckets < 1 || cfg->buckets > 64) return fail(B2R_ERR_ARG, "buckets must be in 1..64");
	if (cfg->max_bounces < 1 || cfg->max_bounces > 1024) return fail(B2R_ERR_ARG, "max_bounces must be in 1..1024");
	if (cfg->bucket_stride > 1 && cfg->bucket_first >= cfg->bucket_stride) return fail(B2R_ERR_ARG, "bucket_first must be < bucket_stride");
	if (cfg->samples_in_flight > static_cast<uint32_t>(kMaxSlots)) return fail(B2R_ERR_ARG, "samples_in_flight must be <= 64");
	if ((cfg->flags & B2R_FLAG_GGX) && (cfg->flags & B2R_FLAG_REFERENCE_EXACT)) return fail(B2R_ERR_ARG, "B2R_FLAG_GGX cannot be combined with B2R_FLAG_REFERENCE_EXACT");
	if ((cfg->flags & B2R_FLAG_DIELECTRIC) && (cfg->flags & B2R_FLAG_REFERENCE_EXACT)) return fail(B2R_ERR_ARG, "B2R_FLAG_DIELECTRIC cannot be combined with B2R_FLAG_REFERENCE_EXACT");
	if (const char* why = sky_flag_conflict(cfg->flags)) return fail(B2R_ERR_ARG, why);
	if (const char* why = light_tree_flag_conflict(cfg->flags)) return fail(B2R_ERR_ARG, why);
	int n_dev = 0;
	cudaError_t e = cudaGetDeviceCount(&n_dev);
	if (e != cudaSuccess || n_dev == 0) return fail(B2R_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libb2r has no CPU fallback)");
	if (cfg->device < 0 || cfg->device >= n_dev) return fail(B2R_ERR_ARG, "device ordinal out of range");
	b2r_ctx* c = new b2r_ctx();
	c->cfg = *cfg;
	c->slots = cfg->samples_in_flight;  // 0 = chosen from the image size in alloc_frame
	c->packet_primary = std::getenv("B2R_NO_PACKET") == nullptr;  // A/B switch for measurements: per-lane walks for the camera rays too
	c->lanes_max = std::getenv("B2R_NO_TWIN") ? 1u : 2u;          // A/B switches for measurements: every batch as one lane / B2R_LANES = 1, 2 or 4
	if (const char* v = std::getenv("B2R_SIDES")) { c->sides = std::atoi(v) == 1 ? 1u : 2u; }   // A/B switch: 1 = every batch on the caller's stream, one after the other
	if (const char* v = std::getenv("B2R_LANES")) { const int n = std::atoi(v); if (n == 1 || n == 2 || n == 4) { c->lanes_max = static_cast<uint32_t>(n); c->lanes_forced = true; } }
	if (const char* v = std::getenv("B2R_LANE_GRID")) { c->lane_grid_frac = static_cast<float>(std::atof(v)); if (!(c->lane_grid_frac > 0.0f && c->lane_grid_frac <= 1.0f)) c->lane_grid_frac = 1.0f; }
	int rc = ensure_device(c);
	if (!rc) { cudaDeviceProp prop; e = cudaGetDeviceProperties(&prop, cfg->device); if (e != cudaSuccess) rc = fail(B2R_ERR_CUDA, cudaGetErrorString(e)); else { c->sm_count = prop.multiProcessorCount; c->grid_stream = c->sm_count * 8; } }
	if (!rc) { e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking); if (e != cudaSuccess) rc = fail(B2R_ERR_CUDA, cudaGetErrorString(e)); c->stream = c->own_stream; }
	if (!rc) rc = alloc_frame(c);
	if (rc) { b2r_destroy(c); return rc; }
	*out = c;
	return B2R_OK;
}

void b2r_destroy(b2r_ctx* c) {
	if (!c) return;
	cudaSetDevice(c->cfg.device);
	if (c->stream) sync_main(c);
	for (size_t r = 0; r < c->peer_acc.size(); r++) if (c->peer_acc[r] && r != c->my_rank) cudaIpcCloseMemHandle(c->peer_acc[r]);
	b2r_team_close(c); if (c->d_team) { cudaFree(c->d_team); c->d_team = nullptr; }
	drop_graph(c);
	for (auto& t : c->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
	free_tables(c->tables);
	dev_free(&c->d_cost); dev_free(&c->d_remap); dev_free(&c->d_trace); dev_free(&c->d_tap); dev_free(&c->d_cost_base); dev_free(&c->d_sort_tmp); dev_free(&c->d_sweep); dev_free(&c->d_sky_tmp);
	for (int k = 0; k < 2; k++) { dev_free(&c->d_mkey[k]); dev_free(&c->d_midx[k]); }
	for (int s = 0; s < 2; s++) { dev_free(&c->d_A[s]); dev_free(&c->d_B[s]); dev_free(&c->d_T[s]); dev_free(&c->d_N[s]); }
	dev_free(&c->d_H); dev_free(&c->d_SA); dev_free(&c->d_SB); dev_free(&c->d_SL); dev_free(&c->d_SS); dev_free(&c->d_rad); dev_free(&c->d_acc); dev_free(&c->d_fb);
	for (int s = 0; s < 2; s++) { dev_free(&c->d_ex_slot[s]); dev_free(&c->d_ex_act[s]); }
	dev_free(&c->d_ex_key); dev_free(&c->d_ex_next);
	dev_free(&c->d_counts); dev_free(&c->d_stats); dev_free(&c->d_batch);
	if (c->h_stage) cudaFreeHost(c->h_stage);
	if (c->ev_stage) cudaEventDestroy(c->ev_stage);
	if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); cudaEventDestroy(c->ev_resolved); cudaEventDestroy(c->ev_copied); }
	free_side_scenes(c);
	if (c->up_stream) { cudaStreamSynchronize(c->up_stream); cudaStreamDestroy(c->up_stream); cudaEventDestroy(c->ev_main_mark); }
	if (c->ev_uploaded) cudaEventDestroy(c->ev_uploaded);
	for (auto& S : c->side) {
		if (S.ev_refreshed) cudaEventDestroy(S.ev_refreshed);
		S.track.destroy();
		if (S.stream) { cudaStreamDestroy(S.stream); cudaEventDestroy(S.ev_traced); cudaEventDestroy(S.ev_folded); cudaEventDestroy(S.ev_sync); }
	}
	c->main.destroy();
	if (c->own_stream) cudaStreamDestroy(c->own_stream);
	delete c;
}

int b2r_resize(b2r_ctx* c, uint32_t width, uint32_t height) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	if (width == 0 || height == 0 || width % 16 || height % 16) return fail(B2R_ERR_ARG, "width/height must be non-zero multiples of 16");
	if (static_cast<uint64_t>(width) * height > kPixMask) return fail(B2R_ERR_ARG, "image too large");
	int rc = ensure_device(c); if (rc) return rc;
	CU(sync_main(c));
	if (c->copy_pending) { CU(cudaEventSynchronize(c->ev_copied)); c->copy_pending = false; }
	if (width == c->cfg.width && height == c->cfg.height) return b2r_reset(c);
	if (!c->peer_acc.empty() || !c->team_acc.empty()) return fail(B2R_ERR_STATE, "the bucket array / framebuffer are exported to peers (CUDA IPC): b2r_ipc_close / b2r_team_close on every rank before a resize, then export again");
	c->cfg.width = width; c->cfg.height = height;
	return alloc_frame(c);
}

int b2r_reset(b2r_ctx* c) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	c->accumulations = 0; drop_speculation(c);
	if ((rc = team_before_bucket_write(c))) return rc;
	const size_t npix = static_cast<size_t>(c->cfg.width) * c->cfg.height;
	CU(cudaMemsetAsync(c->d_acc, 0, static_cast<size_t>(c->cfg.buckets) * 3 * npix * sizeof(float), c->stream));
	return B2R_OK;
}

int b2r_set_stream(b2r_ctx* c, void* cuda_stream) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	CU(sync_main(c));
	c->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : c->own_stream;
	drop_graph(c);
	return B2R_OK;
}

int b2r_sync(b2r_ctx* c) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	CU(sync_main(c));
	return collect_timings(c);
}

int b2r_set_flags(b2r_ctx* c, uint32_t flags) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	CU(sync_main(c));
	if ((c->cfg.flags ^ flags) & B2R_FLAG_REFERENCE_TREE) return fail(B2R_ERR_STATE, "B2R_FLAG_REFERENCE_TREE can only be chosen at b2r_create");
	if ((c->cfg.flags ^ flags) & B2R_FLAG_REFERENCE_EXACT) return fail(B2R_ERR_STATE, "B2R_FLAG_REFERENCE_EXACT can only be chosen at b2r_create");
	if ((flags & B2R_FLAG_GGX) && (flags & B2R_FLAG_REFERENCE_EXACT)) return fail(B2R_ERR_ARG, "B2R_FLAG_GGX cannot be combined with B2R_FLAG_REFERENCE_EXACT");
	if ((flags & B2R_FLAG_DIELECTRIC) && (flags & B2R_FLAG_REFERENCE_EXACT)) return fail(B2R_ERR_ARG, "B2R_FLAG_DIELECTRIC cannot be combined with B2R_FLAG_REFERENCE_EXACT");
	if ((flags & B2R_FLAG_DIELECTRIC) && c->have_scene && !c->scene_diel_valid) return fail(B2R_ERR_ARG, kDielInvalid);
	if (const char* why = sky_flag_conflict(flags)) return fail(B2R_ERR_ARG, why);
	if (const char* why = light_tree_flag_conflict(flags)) return fail(B2R_ERR_ARG, why);
	if ((flags & B2R_FLAG_LIGHT_TREE) && c->have_scene && !c->lt_valid) return fail(B2R_ERR_ARG, kLightsInvalid);
	const SceneDev& sc = c->params.scene;
	if ((flags & B2R_FLAG_SKY_LIGHT) && c->have_scene && sc.has_ambient && !c->sky_checked) {  // uploaded without the flag: the rule is checked on the texels now
		std::vector<float4> tex(c->hdri_texels);
		CU(cudaMemcpyAsync(tex.data(), c->tables.hdri.p, tex.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream)); CU(sync_main(c));
		c->sky_valid = sky_texels_valid(tex.data(), tex.size(), sc.ambient, &c->sky_nonzero); c->sky_checked = true;
	}
	if ((flags & B2R_FLAG_SKY_LIGHT) && c->have_scene && sc.has_ambient && !c->sky_valid) return fail(B2R_ERR_ARG, kSkyInvalid);
	if (c->have_scene && sky_sampled(c, flags) && !c->sky_built) {  // turned on over a sky: its tables, from the device copy of the texture
		size_t len[LEN_COUNT] = {}; sky_table_lens(sc.hdri_w, sc.hdri_h, len);
		if ((rc = reserve_tables(c, len)) || (rc = begin_scene_write(c, use_sides(c))) || (rc = launch_sky_build(c, sc.hdri_w, sc.hdri_h, sc.ambient)) || (rc = end_scene_write(c))) return rc;
		c->sky_built = true; bind_tables(c->params, c->tables, sc.hdri != nullptr);
	}
	if ((flags & B2R_FLAG_LIGHT_TREE) && c->have_scene && !c->lt_built) {  // turned on over a scene: the tree, over the device's BVH-order spheres
		std::vector<float4> prims(sc.n_prims); std::vector<int32_t> prim_mat(sc.n_prims);
		CU(cudaMemcpyAsync(prims.data(), c->tables.prims.p, prims.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
		CU(cudaMemcpyAsync(prim_mat.data(), c->tables.prim_mat.p, prim_mat.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream)); CU(sync_main(c));
		LightTree lt; size_t len[LEN_COUNT] = {}; build_kept_light_tree(c, prims.data(), prim_mat.data(), sc.n_prims, lt, len);
		if ((rc = reserve_tables(c, len)) || (rc = begin_scene_write(c, use_sides(c)))) return rc;
		const UploadPart parts[] = {{c->tables.ltree_nodes.p, lt.nodes.data(), lt.nodes.size() * sizeof(float4)}, {c->tables.ltree_light.p, lt.light.data(), lt.light.size() * sizeof(int4)},
		                            {c->tables.ltree_prim_light.p, lt.prim_light.data(), lt.prim_light.size() * sizeof(int32_t)}};
		if ((rc = stage_upload(c, parts, 3)) || (rc = end_scene_write(c))) return rc;
		c->lt_built = true; c->lt_nodes = static_cast<uint32_t>(lt.nodes.size() / 2u); bind_tables(c->params, c->tables, sc.hdri != nullptr);
	}
	c->cfg.flags = flags; c->params.frame.flags = flags;
	set_sky_scalars(c);
	if (c->have_scene) {
		const uint32_t n = c->params.scene.n_prims;
		c->use_bvh = (flags & B2R_FLAG_FORCE_BVH) ? true : (flags & B2R_FLAG_FORCE_BRUTE) ? false : n > 32;
	}
	drop_graph(c);
	return B2R_OK;
}

} // extern "C"
namespace {
// Host arrays -> device through ONE page-locked block, without stream synchronisation: the copies are ordered after the kernels
// already enqueued (which may still read the old scene) and before the ones enqueued next; the block is only rewritten once the
// previous upload's copies have completed (an event early in the previous frame, not its end).
int stage_upload(b2r_ctx* c, const UploadPart* parts, size_t n_parts) {
	size_t total = 0; for (size_t i = 0; i < n_parts; i++) total += (parts[i].bytes + 255) & ~static_cast<size_t>(255);
	if (c->stage_busy) { CU(cudaEventSynchronize(c->ev_stage)); c->stage_busy = false; }
	if (total > c->stage_bytes) {
		if (c->h_stage) CU(cudaFreeHost(c->h_stage));
		c->h_stage = nullptr; c->stage_bytes = 0;
		CU(cudaMallocHost(reinterpret_cast<void**>(&c->h_stage), total)); c->stage_bytes = total;
	}
	if (!c->ev_stage) CU(cudaEventCreateWithFlags(&c->ev_stage, cudaEventDisableTiming));
	size_t off = 0;
	for (size_t i = 0; i < n_parts; i++) {
		const UploadPart& q = parts[i];
		if (q.bytes) { std::memcpy(c->h_stage + off, q.src, q.bytes); CU(cudaMemcpyAsync(q.dst, c->h_stage + off, q.bytes, cudaMemcpyHostToDevice, c->scene_st)); }
		off += (q.bytes + 255) & ~static_cast<size_t>(255);
	}
	CU(cudaEventRecord(c->ev_stage, c->scene_st)); c->stage_busy = true;
	return B2R_OK;
}
// stage_upload of the tables pack_scene fills (into the primary tables, list order), then `extra`
int stage_packed(b2r_ctx* c, const PackedScene& ps, std::initializer_list<UploadPart> extra) {
#define X(T, name, len) {c->tables.name.p, ps.name.data(), ps.name.size() * sizeof(T)},
	std::vector<UploadPart> parts = {B2R_PACKED_TABLES(X)};
#undef X
	parts.insert(parts.end(), extra);
	return stage_upload(c, parts.data(), parts.size());
}
// What b2r_upload_scene and b2r_refit_scene both check: material and light indices in range, and B2R_FLAG_DIELECTRIC's rule on the
// materials (*diel_valid: whether they follow it, for a later b2r_set_flags).
int check_scene_refs(const b2r_ctx* c, const b2r_sphere* prims, const b2r_sphere* geometry, uint32_t n_prims, uint32_t n_geom, const b2r_material* materials, uint32_t n_mat,
                     const int32_t* light_geom_idx, uint32_t n_lights, bool* diel_valid) {
	for (uint32_t i = 0; i < n_prims; i++) if (prims[i].material_ID < 0 || static_cast<uint32_t>(prims[i].material_ID) >= n_mat || geometry[i].material_ID < 0 || static_cast<uint32_t>(geometry[i].material_ID) >= n_mat) return fail(B2R_ERR_ARG, "material_ID out of range");
	for (uint32_t i = 0; i < n_lights; i++) if (light_geom_idx[i] < 0 || static_cast<uint32_t>(light_geom_idx[i]) >= n_geom) return fail(B2R_ERR_ARG, "light index out of range");
	*diel_valid = dielectric_materials_valid(materials, n_mat);
	if (!*diel_valid && (c->cfg.flags & B2R_FLAG_DIELECTRIC)) return fail(B2R_ERR_ARG, kDielInvalid);
	return B2R_OK;
}
// After a scene write: the kernels' parameter block points at the primary tables (`sky`: hdri too) and `set` writes the scene's scalars
// into it. The captured graphs hold that block by value and run one pipeline: they are dropped when either changed.
template <typename F> void rebind_scene(b2r_ctx* c, bool sky, F&& set) {
	const Params before = c->params; const bool bvh_before = c->use_bvh;
	bind_tables(c->params, c->tables, sky);
	set(c->params.scene);
	set_sky_scalars(c);
	if (!c->have_scene || bvh_before != c->use_bvh || std::memcmp(&before, &c->params, sizeof before) != 0) drop_graph(c);
}
}  // namespace
extern "C" {

int b2r_upload_scene(b2r_ctx* c, const b2r_sphere* prims, const b2r_bvh_node* nodes, uint32_t n_prims, uint32_t n_nodes,
                     const b2r_material* materials, uint32_t n_mat, const int32_t* light_geom_idx, uint32_t n_lights,
                     const b2r_sphere* geometry, uint32_t n_geom, const float ambient[3], const float* hdri_rgba, int32_t hdri_w, int32_t hdri_h) {
	if (!c || !prims || !nodes || !materials || !geometry || n_prims == 0 || n_mat == 0) return fail(B2R_ERR_ARG, "null or empty scene array");
	if (n_geom != n_prims) return fail(B2R_ERR_ARG, "geometry and BVH-order primitive counts differ");
	if (n_lights && !light_geom_idx) return fail(B2R_ERR_ARG, "null light list");
	if (!validate_reference_bvh(nodes, n_nodes, n_prims)) return fail(B2R_ERR_BVH, "node array is not a 2n-1 binary tree with adjacent children and single-sphere leaves");
	const float amb[3] = {ambient ? ambient[0] : 0.0f, ambient ? ambient[1] : 0.0f, ambient ? ambient[2] : 0.0f};
	const bool has_ambient = sel_max(amb[0], sel_max(amb[1], amb[2])) > 0.0f;
	if (has_ambient && (!hdri_rgba || hdri_w <= 0 || hdri_h <= 0)) return fail(B2R_ERR_ARG, "ambient > 0 needs an HDRI (the reference terminates without one, Application.cpp:225-229)");
	bool diel_valid = true;
	int rc = check_scene_refs(c, prims, geometry, n_prims, n_geom, materials, n_mat, light_geom_idx, n_lights, &diel_valid); if (rc) return rc;
	// B2R_FLAG_SKY_LIGHT: the input rule on the sky's texels, checked here under the flag (otherwise when b2r_set_flags turns it on)
	const bool sky_checked = (c->cfg.flags & B2R_FLAG_SKY_LIGHT) && has_ambient;
	bool sky_nonzero = false;
	if (sky_checked && !sky_texels_valid(reinterpret_cast<const float4*>(hdri_rgba), static_cast<size_t>(hdri_w) * hdri_h, amb, &sky_nonzero)) return fail(B2R_ERR_ARG, kSkyInvalid);
	const bool sky_build = sky_checked && sky_nonzero;
	// B2R_FLAG_LIGHT_TREE: the input rule on the light list, refused here under the flag (otherwise when b2r_set_flags turns it on)
	const bool lt_build = (c->cfg.flags & B2R_FLAG_LIGHT_TREE) != 0, lt_valid = light_list_valid(materials, light_geom_idx, n_lights, geometry);
	if (lt_build && !lt_valid) return fail(B2R_ERR_ARG, kLightsInvalid);
	if ((rc = ensure_device(c))) return rc;
	// No stream synchronisation from here on: the copies below are ordered after the kernels already enqueued on the stream (which
	// may still read the old scene) and before the ones enqueued next. The host side is staged in one page-locked block that is only
	// rewritten once the previous upload's copies have completed (an event early in the previous frame, not its end).

	const bool gpu_tree = (c->cfg.flags & B2R_FLAG_GPU_TREE) && !(c->cfg.flags & B2R_FLAG_REFERENCE_TREE);
	if (gpu_tree) {
		// the tree is built on the device below (after the spheres have been copied): only its shape is worked out here
		float lo[3], hi[3]; sphere_bounds(prims, n_prims, lo, hi);
		const float corners[6] = {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]};
		float cam[6]; const uint32_t n_cam = camera_origins(c, cam);
		if (!c->obox_valid || !origin_box_holds(c->obox, corners, 2) || !origin_box_holds(c->obox, cam, n_cam))
			{ c->obox = origin_box_rule(lo, hi, cam, n_cam); c->obox_valid = true; }
		for (int k = 0; k < 3; k++) { c->sph_lo[k] = lo[k]; c->sph_hi[k] = hi[k]; c->wide_host.sphere_lo[k] = lo[k]; c->wide_host.sphere_hi[k] = hi[k]; }
		WideBvh& w = c->wide_host;
		w.nodes.clear(); w.prims.clear(); w.geom_of_prim.clear(); w.cost = 0.0; w.ob = c->obox;
		packed_levels(n_prims, w.level_first);
		w.depth = static_cast<uint32_t>(w.level_first.size()) - 1u; w.max_stack = 3u * w.depth;
		c->n_wide = w.level_first.back();
		uint32_t node_bits = 1; while ((1ull << node_bits) < c->n_wide) node_bits++;
		w.tn_bits = 32u - node_bits < 29u ? 32u - node_bits : 29u;
		if ((c->cfg.flags & (B2R_FLAG_GPU_SAH | B2R_FLAG_GPU_SAH3)) && n_prims >= 2u && n_prims > c->n_wide) c->n_wide = n_prims;  // the sweep tree: fewer nodes than spheres, how many is known once it is built (reserve for the bound)
		c->wide_key = 0; c->wide_blob.clear(); c->have_wide = true; c->gpu_tree = true;
		c->lazy_prims.assign(prims, prims + n_prims); c->lazy_geom.assign(geometry, geometry + n_geom);  // matched by value only if a refit ever asks
	} else {
	{  // derived traversal layout, cached on everything it is derived from: the 20 meaningful bytes of every sphere (and, for the
			// reference topology, the node array); a hit is confirmed by comparing the kept copies, not just the hash
			auto fnv = [](uint64_t h, const void* data, size_t bytes) { const unsigned char* b = static_cast<const unsigned char*>(data); for (size_t i = 0; i < bytes; i++) h = (h ^ b[i]) * 1099511628211ull; return h; };
			const bool ref_tree = (c->cfg.flags & B2R_FLAG_REFERENCE_TREE) != 0;
			uint64_t key = 1469598103934665603ull ^ (ref_tree ? 0x9e3779b97f4a7c15ull : 0ull);
			std::vector<unsigned char> blob(static_cast<size_t>(n_prims) * 20 + (ref_tree ? static_cast<size_t>(n_nodes) * sizeof(b2r_bvh_node) : 0));
			for (uint32_t i = 0; i < n_prims; i++) std::memcpy(blob.data() + static_cast<size_t>(i) * 20, &prims[i], 20);
			if (ref_tree) std::memcpy(blob.data() + static_cast<size_t>(n_prims) * 20, nodes, static_cast<size_t>(n_nodes) * sizeof(b2r_bvh_node));
			key = fnv(key, blob.data(), blob.size());
			const bool same_tree = c->have_wide && key == c->wide_key && blob == c->wide_blob;
			float lo[3], hi[3]; sphere_bounds(prims, n_prims, lo, hi);
			// the origin box is kept while it still holds the spheres and the camera; a different scene starts from a fresh one
			const float corners[6] = {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]};
			float cam[6]; const uint32_t n_cam = camera_origins(c, cam);
			if (!same_tree || !c->obox_valid || !origin_box_holds(c->obox, corners, 2) || !origin_box_holds(c->obox, cam, n_cam))
				{ c->obox = origin_box_rule(lo, hi, cam, n_cam); c->obox_valid = true; }
			for (int k = 0; k < 3; k++) { c->sph_lo[k] = lo[k]; c->sph_hi[k] = hi[k]; }
			if (!same_tree) {
				if (ref_tree) flatten_bvh(nodes, n_nodes, prims, n_prims, c->wide_host, &c->obox);
				else { std::vector<b2r_bvh_node> tree; build_traversal_tree(prims, n_prims, tree); flatten_bvh(tree.data(), static_cast<uint32_t>(tree.size()), prims, n_prims, c->wide_host, &c->obox); }
				c->wide_key = key; c->wide_blob.swap(blob); c->have_wide = true;
				match_prims_to_geometry(prims, geometry, n_prims, c->wide_host.geom_of_prim);  // which sphere each leaf stands for (b2r_refit_scene); left empty if prims is no permutation of geometry
			} else if (std::memcmp(&c->wide_host.ob, &c->obox, sizeof(OriginBox)) != 0) wide_fill_boxes(c->wide_host, c->wide_host.prims.data(), c->obox);  // same topology, boxes for the current origin box
		}
		c->gpu_tree = false; c->n_wide = static_cast<uint32_t>(c->wide_host.nodes.size());
	}
	if (c->wide_host.max_stack + 3u > static_cast<uint32_t>(kTraversalStack)) { c->have_wide = false; return fail(B2R_ERR_BVH, "tree needs a deeper traversal stack than kTraversalStack (3 slots of headroom for the branch-free pushes)"); }
	if (c->n_wide >= kMaxWideNodes) { c->have_wide = false; return fail(B2R_ERR_BVH, "more than 2^22 traversal nodes (stack entries keep 22 node bits)"); }

	PackedScene ps; pack_scene(prims, n_prims, materials, n_mat, light_geom_idx, n_lights, geometry, ps);
	const size_t texels = has_ambient ? static_cast<size_t>(hdri_w) * hdri_h : 0;
	size_t len[LEN_COUNT] = {n_prims, n_mat, ps.light_sphere.size(), c->n_wide, texels, 0, 0, 0};  // (no sky: the sky's tables are left alone)
	if (sky_build) sky_table_lens(hdri_w, hdri_h, len);
	keep_light_list(c, materials, light_geom_idx, n_lights, geometry, lt_valid);
	LightTree lt; if (lt_build) build_kept_light_tree(c, ps.prims.data(), ps.prim_mat.data(), n_prims, lt, len);
	if ((rc = reserve_tables(c, len))) return rc;
	const bool bvh_next = (c->cfg.flags & B2R_FLAG_FORCE_BVH) ? true : (c->cfg.flags & B2R_FLAG_FORCE_BRUTE) ? false : n_prims > 32;
	if ((rc = begin_scene_write(c, sides_for(c, bvh_next)))) return rc;
	if ((rc = stage_packed(c, ps, {{c->tables.wide.p, c->wide_host.nodes.data(), gpu_tree ? 0 : c->wide_host.nodes.size() * sizeof(WideNode)}, {c->tables.hdri.p, hdri_rgba, texels * sizeof(float4)},
	                               {c->tables.ltree_nodes.p, lt.nodes.data(), lt.nodes.size() * sizeof(float4)}, {c->tables.ltree_light.p, lt.light.data(), lt.light.size() * sizeof(int4)},
	                               {c->tables.ltree_prim_light.p, lt.prim_light.data(), lt.prim_light.size() * sizeof(int32_t)}}))) return rc;
	c->hdri_texels = texels; c->lt_built = lt_build; c->lt_nodes = static_cast<uint32_t>(lt.nodes.size() / 2u);
	if (sky_build && (rc = launch_sky_build(c, hdri_w, hdri_h, amb))) return rc;
	c->sky_built = sky_build; c->sky_checked = sky_checked; c->sky_valid = true; c->sky_nonzero = sky_nonzero;
	c->wide_refit = false; c->cur_geom_of_prim.clear(); drop_speculation(c);
	if (gpu_tree) {  // Morton keys -> stable radix sort -> implicit 4-ary links -> boxes, all on the stream behind the copies above
		if (n_prims > c->cap_mkey) { for (int k = 0; k < 2; k++) { size_t cap = 0; if ((rc = dev_reserve(&c->d_mkey[k], &cap, n_prims)) || (cap = 0, rc = dev_reserve(&c->d_midx[k], &cap, n_prims))) return rc; } c->cap_mkey = n_prims; }
		float scale[3]; morton_scale(c->sph_lo, c->sph_hi, scale);
		k_morton_keys<<<(n_prims + kBlock - 1u) / kBlock, kBlock, 0, c->scene_st>>>(c->tables.prims.p, n_prims, c->sph_lo[0], c->sph_lo[1], c->sph_lo[2], scale[0], scale[1], scale[2], c->d_mkey[0], c->d_midx[0]);
		size_t tmp = 0;
		CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp, c->d_mkey[0], c->d_mkey[1], c->d_midx[0], c->d_midx[1], static_cast<int>(n_prims), 0, 30, c->scene_st));
		if ((rc = dev_reserve(&c->d_sort_tmp, &c->cap_sort_tmp, tmp))) return rc;
		CU(cub::DeviceRadixSort::SortPairs(c->d_sort_tmp, tmp, c->d_mkey[0], c->d_mkey[1], c->d_midx[0], c->d_midx[1], static_cast<int>(n_prims), 0, 30, c->scene_st));
		bool swept = false;
		if ((c->cfg.flags & (B2R_FLAG_GPU_SAH | B2R_FLAG_GPU_SAH3)) && n_prims >= 2u && (rc = sweep_build(c, (c->cfg.flags & B2R_FLAG_GPU_SAH3) ? nullptr : c->d_midx[1], n_prims, &swept))) return rc;
		if (!swept) {
			c->n_wide = c->wide_host.level_first.back();  // (the packed shape worked out above)
			PackedLevels lv{}; lv.levels = c->wide_host.depth;
			if (lv.levels + 1u > sizeof lv.first / sizeof lv.first[0]) return fail(B2R_ERR_BVH, "packed tree deeper than 23 levels");
			for (uint32_t l = 0; l <= lv.levels; l++) lv.first[l] = c->wide_host.level_first[l];
			k_packed_links<<<(c->n_wide * 4u + kBlock - 1u) / kBlock, kBlock, 0, c->scene_st>>>(reinterpret_cast<float4*>(c->tables.wide.p), lv, n_prims, c->d_midx[1]);
			c->launches++;
		}
		CU(cudaGetLastError()); c->launches += 2;
		if ((rc = launch_refit_levels(c, nullptr))) return rc;
		if (!c->d_cost_base) { size_t cap = 0; if ((rc = dev_reserve(&c->d_cost_base, &cap, 1))) return rc; }
		CU(cudaMemsetAsync(c->d_cost_base, 0, sizeof(double), c->scene_st));
		k_tree_cost<<<c->sm_count * 4, kBlock, 0, c->scene_st>>>(reinterpret_cast<const float4*>(c->tables.wide.p), c->n_wide, c->d_cost_base);  // what a later refit's quality ratio is measured against
		c->launches++;
		c->wide_refit = true;  // the device holds the only copy of this tree
	}
	if ((rc = launch_link_tables(c))) return rc;
	if ((rc = end_scene_write(c))) return rc;
	rebind_scene(c, has_ambient, [&](SceneDev& s) {
		s.n_prims = n_prims; s.n_mat = n_mat; s.n_lights = n_lights; s.stack_tn_bits = c->wide_host.tn_bits;
		s.light_sel_pdf = n_lights ? 1.0f / static_cast<float>(n_lights) : 0.0f;  // Renderer.hpp:78 (no lights: Q15, light sampling is skipped and the MIS weight of an emissive hit is 1)
		s.ambient[0] = amb[0]; s.ambient[1] = amb[1]; s.ambient[2] = amb[2]; s.has_ambient = has_ambient ? 1 : 0;
		s.hdri_w = hdri_w; s.hdri_h = hdri_h; s.hdri_fw = static_cast<float>(hdri_w - 1); s.hdri_fh = static_cast<float>(hdri_h - 1);  // Application.cpp:230-231
		c->use_bvh = bvh_next;
	});
	c->have_scene = true; c->scene_diel_valid = diel_valid;
	return B2R_OK;
}

int b2r_refit_scene(b2r_ctx* c, const b2r_sphere* prims, uint32_t n_prims, const b2r_material* materials, uint32_t n_mat,
                    const int32_t* light_geom_idx, uint32_t n_lights, const b2r_sphere* geometry, uint32_t n_geom, float* quality_out) {
	if (!c || !prims || !materials || !geometry || n_prims == 0 || n_mat == 0) return fail(B2R_ERR_ARG, "null or empty scene array");
	if (!c->have_scene || !c->have_wide) return fail(B2R_ERR_STATE, "b2r_refit_scene needs the topology of an earlier b2r_upload_scene");
	if (n_prims != c->params.scene.n_prims || n_geom != n_prims) return fail(B2R_ERR_ARG, "a refit keeps the sphere count (and BVH order) of the last b2r_upload_scene");
	if (n_lights && !light_geom_idx) return fail(B2R_ERR_ARG, "null light list");
	bool diel_valid = true;
	int rc = check_scene_refs(c, prims, geometry, n_prims, n_geom, materials, n_mat, light_geom_idx, n_lights, &diel_valid); if (rc) return rc;
	const bool lt_build = (c->cfg.flags & B2R_FLAG_LIGHT_TREE) != 0, lt_valid = light_list_valid(materials, light_geom_idx, n_lights, geometry);
	if (lt_build && !lt_valid) return fail(B2R_ERR_ARG, kLightsInvalid);
	if ((rc = ensure_device(c))) return rc;
	// The caller may have re-sorted its prims (the reference's constructor does on every rebuild, BVH.hpp:201-205): leaf links become
	// indices into the NEW order. old index -> geometry index (known from the last upload / refit) -> new index (matched by value).
	if (c->gpu_tree && c->wide_host.geom_of_prim.empty() && c->lazy_prims.size() == n_prims)  // a device-built tree: which sphere each leaf stands for is worked out on the first refit
		match_prims_to_geometry(c->lazy_prims.data(), c->lazy_geom.data(), n_prims, c->wide_host.geom_of_prim);
	const std::vector<uint32_t>& old_geom = c->cur_geom_of_prim.empty() ? c->wide_host.geom_of_prim : c->cur_geom_of_prim;
	if (old_geom.size() != n_prims) return fail(B2R_ERR_STATE, "the uploaded prims were not a permutation of geometry: no refit for this scene");
	std::vector<uint32_t> new_geom, remap;
	bool same_order = true;  // the cheap case first: the caller kept its leaf order (one sequential pass instead of a hash table)
	for (uint32_t i = 0; i < n_prims && same_order; i++) same_order = std::memcmp(&prims[i], &geometry[old_geom[i]], 20) == 0;
	if (!same_order) {
		if (!match_prims_to_geometry(prims, geometry, n_prims, new_geom)) return fail(B2R_ERR_ARG, "prims_bvh_order is not a permutation of geometry");
		same_order = new_geom == old_geom;
	}
	if (!same_order) {
		std::vector<uint32_t> prim_of_geom(n_prims);
		for (uint32_t i = 0; i < n_prims; i++) prim_of_geom[new_geom[i]] = i;
		remap.resize(n_prims);
		for (uint32_t i = 0; i < n_prims; i++) remap[i] = prim_of_geom[old_geom[i]];
	}
	PackedScene ps; pack_scene(prims, n_prims, materials, n_mat, light_geom_idx, n_lights, geometry, ps);
	if ((rc = dev_reserve(&c->d_remap, &c->cap_remap, remap.size()))) return rc;
	size_t len[LEN_COUNT] = {0, n_mat, ps.light_sphere.size(), 0, 0, 0, 0, 0};  // the sphere count is kept: only the (small) material and light tables can grow
	keep_light_list(c, materials, light_geom_idx, n_lights, geometry, lt_valid);
	LightTree lt; if (lt_build) build_kept_light_tree(c, ps.prims.data(), ps.prim_mat.data(), n_prims, lt, len);  // (the light list, and perhaps the BVH order, changed)
	if ((rc = reserve_tables(c, len))) return rc;
	if (!c->d_cost) { size_t cap = 0; if ((rc = dev_reserve(&c->d_cost, &cap, 1))) return rc; }
	if ((rc = begin_scene_write(c, use_sides(c)))) return rc;
	if ((rc = stage_packed(c, ps, {{c->d_remap, remap.data(), remap.size() * sizeof(uint32_t)},
	                               {c->tables.ltree_nodes.p, lt.nodes.data(), lt.nodes.size() * sizeof(float4)}, {c->tables.ltree_light.p, lt.light.data(), lt.light.size() * sizeof(int4)},
	                               {c->tables.ltree_prim_light.p, lt.prim_light.data(), lt.prim_light.size() * sizeof(int32_t)}}))) return rc;
	c->lt_built = lt_build; c->lt_nodes = static_cast<uint32_t>(lt.nodes.size() / 2u);
	if (!same_order) c->cur_geom_of_prim.swap(new_geom);
	// boxes bottom-up on the device, for an origin box that holds the moved spheres
	{
		float lo[3], hi[3]; sphere_bounds(prims, n_prims, lo, hi);
		for (int k = 0; k < 3; k++) { c->sph_lo[k] = lo[k]; c->sph_hi[k] = hi[k]; }
		const float corners[6] = {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]};
		float cam[6]; const uint32_t n_cam = camera_origins(c, cam);
		if (!c->obox_valid || !origin_box_holds(c->obox, corners, 2)) {
			c->obox = origin_box_rule(lo, hi, cam, n_cam); c->obox_valid = true;
			if (!c->gpu_tree) wide_fill_boxes(c->wide_host, c->wide_host.prims.data(), c->obox);  // the as-built tree (reference cost) for the same origin box
		}
	}
	if ((rc = launch_refit_levels(c, same_order ? nullptr : c->d_remap))) return rc;
	if (!same_order && (rc = launch_link_tables(c))) return rc;  // leaves were re-linked into the new BVH order
	if ((rc = end_scene_write(c))) return rc;
	c->wide_refit = true; drop_speculation(c); c->scene_diel_valid = diel_valid;
	rebind_scene(c, c->params.scene.hdri != nullptr, [&](SceneDev& s) {
		s.n_mat = n_mat; s.n_lights = n_lights; s.light_sel_pdf = n_lights ? 1.0f / static_cast<float>(n_lights) : 0.0f;  // Renderer.hpp:78
	});
	if (quality_out) {  // optional: costs one launch and a stream synchronisation
		c->main_reads_scene = true;
		CU(cudaMemsetAsync(c->d_cost, 0, sizeof(double), c->stream));
		k_tree_cost<<<c->sm_count * 4, kBlock, 0, c->stream>>>(reinterpret_cast<const float4*>(c->tables.wide.p), c->n_wide, c->d_cost);
		c->launches++;
		double cost = 0.0, base = c->wide_host.cost;
		CU(cudaMemcpyAsync(&cost, c->d_cost, sizeof cost, cudaMemcpyDeviceToHost, c->stream));
		if (c->gpu_tree && c->d_cost_base) CU(cudaMemcpyAsync(&base, c->d_cost_base, sizeof base, cudaMemcpyDeviceToHost, c->stream));
		CU(sync_main(c));
		*quality_out = base > 0.0 ? static_cast<float>(cost / base) : 1.0f;
	}
	return B2R_OK;
}

int b2r_set_camera(b2r_ctx* c, const float pos[3], const float q[4], float half_width, float half_height, float z, float exposure) {
	if (!c || !pos || !q) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	// the camera travels with every batch's descriptor (k_set_batch, stream-ordered: batches already enqueued keep theirs), so a camera
	// move needs no synchronisation and leaves the captured batch graph alone
	CameraParams cam = c->params.frame.cam;
	cam.px = pos[0]; cam.py = pos[1]; cam.pz = pos[2]; cam.qw = q[0]; cam.qx = q[1]; cam.qy = q[2]; cam.qz = q[3];
	cam.half_width = half_width; cam.half_height = half_height; cam.z = z; cam.exposure = exposure;
	if (!c->have_camera || std::memcmp(&cam, &c->params.frame.cam, sizeof cam) != 0) { c->params.frame.cam = cam; drop_speculation(c); }  // samples traced ahead saw the old camera
	c->have_camera = true;
	c->cam_pos[0] = pos[0]; c->cam_pos[1] = pos[1]; c->cam_pos[2] = pos[2];
	float pts[6]; const uint32_t n_pts = camera_origins(c, pts);
	if (c->have_scene) return ensure_origin_box(c, pts, n_pts);
	return B2R_OK;
}

int b2r_set_lens(b2r_ctx* c, float lens_radius, float focus_distance) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	if (!(lens_radius >= 0.0f && lens_radius <= FLT_MAX)) return fail(B2R_ERR_ARG, "lens_radius must be finite and >= 0");
	if (!(focus_distance > 0.0f && focus_distance <= FLT_MAX)) return fail(B2R_ERR_ARG, "focus_distance must be finite and > 0");
	if (c->cfg.flags & B2R_FLAG_REFERENCE_EXACT) return fail(B2R_ERR_STATE, "B2R_FLAG_REFERENCE_EXACT reproduces the reference's pinhole camera: no lens");
	int rc = ensure_device(c); if (rc) return rc;
	// the lens travels with every batch's descriptor as the camera does; switching between pinhole and lens switches the bounce-0 kernels,
	// which are part of the captured graph
	const LensParams lens{lens_radius, focus_distance};
	if (std::memcmp(&lens, &c->lens, sizeof lens) != 0) {
		const bool switched = (lens_radius > 0.0f) != (c->lens.radius > 0.0f);
		c->lens = lens;
		if (switched) drop_graph(c); else drop_speculation(c);  // samples traced ahead saw the old lens
	}
	float cam[6]; const uint32_t n_cam = camera_origins(c, cam);
	if (c->have_scene) return ensure_origin_box(c, cam, n_cam);
	return B2R_OK;
}

int b2r_accumulate(b2r_ctx* c, uint32_t n_samples) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	if (!c->have_scene || !c->have_camera) return fail(B2R_ERR_STATE, "upload_scene and set_camera must precede accumulate");
	int rc = ensure_device(c); if (rc) return rc;
	if ((rc = team_before_bucket_write(c))) return rc;
	const bool speculate = c->cfg.bucket_stride <= 1 && !(c->cfg.flags & (B2R_FLAG_NO_SPECULATION | B2R_FLAG_NO_GRAPH));
	BatchArgs args; args.n = 0;
	for (uint32_t s = 0; s < n_samples; s++) {
		const uint32_t acc = ++c->accumulations;  // pre-increment: the first sample has index 1 (Renderer.hpp:74, Q1)
		if (c->spec_used < c->spec_count && acc == c->spec_first + c->spec_used) {
			// traced ahead by an earlier call: fold it (samples are folded in index order: earlier samples of this call go first)
			if (args.n) { if ((rc = run_batch(c, args))) return rc; args.n = 0; }
			BatchArgs f = c->spec_args; f.fold = 1ull << f.slot_of(c->spec_used);
			if (use_sides(c)) {  // the samples wait in the side's part of RAD that traced them; that side is not reused before this fold has run
				b2r_ctx::Side& S = c->side[c->spec_side];
				k_set_batch<<<1, kMaxSlots, 0, c->stream>>>(c->d_batch + c->spec_side * (1u + kMaxLanes), f);
				k_accumulate<<<c->grid_stream, kBlock, 0, c->stream>>>(side_params(c, c->spec_side));
				CU(cudaEventRecord(S.ev_folded, c->stream)); S.folded_valid = true;
			} else {
				k_set_batch<<<1, kMaxSlots, 0, c->stream>>>(c->d_batch, f);
				k_accumulate<<<c->grid_stream, kBlock, 0, c->stream>>>(c->params);
			}
			CU(cudaGetLastError()); c->launches += 1;
			if (++c->spec_used == c->spec_count) { c->spec_count = 0; c->spec_used = 0; c->spec_width = c->spec_width * 2u > kSpecMax ? kSpecMax : c->spec_width * 2u; }
			continue;
		}
		if (c->spec_count) drop_speculation(c);  // the caller jumped elsewhere
		if (!owns_sample(c, acc)) continue;
		if (speculate && n_samples == 1) {
			// the reference's frame loop: one Accumulate() per application frame. Trace spec_width samples now, fold the first.
			const uint32_t w = c->spec_width < batch_cap(c) ? c->spec_width : batch_cap(c);
			args.n = w; for (uint32_t i = 0; i < w; i++) args.acc[i] = acc + i;
			args.fold = 1ull;
			if ((rc = run_batch(c, args))) return rc;
			if (w > 1) { c->spec_args = args; c->spec_first = acc; c->spec_count = w; c->spec_used = 1; c->spec_side = c->last_side; }
			else c->spec_width = 2;
			return B2R_OK;
		}
		args.acc[args.n++] = acc;
		if (args.n == batch_cap(c) || (s + 1 == n_samples && args.n)) { if ((rc = run_batch(c, args))) return rc; args.n = 0; }
	}
	if (args.n) { if ((rc = run_batch(c, args))) return rc; }
	return B2R_OK;
}

static int resolve_with(b2r_ctx* c, const BucketPtrs& bp, float* rgba_out_host, int tonemap, bool async = false, bool enqueue_only = false) {
	int rc = ensure_device(c); if (rc) return rc;
	if (c->accumulations == 0 || c->accumulations % c->cfg.buckets) return B2R_ERR_NOT_READY;  // Renderer.hpp:437
	const float scale = c->params.frame.cam.exposure / static_cast<float>(c->accumulations / c->cfg.buckets);  // :439
	const bool profile = (c->cfg.flags & B2R_FLAG_NO_GRAPH) != 0;
	if (c->copy_pending) CU(cudaStreamWaitEvent(c->stream, c->ev_copied, 0));  // the previous frame is still being read out of d_fb
	rc = launch(c, KK_RESOLVE, profile, [&] { k_resolve<<<c->grid_stream, kBlock, 0, c->stream>>>(c->params.frame, bp, c->d_fb, scale, tonemap, 0u, c->params.frame.npix); });
	if (rc) return rc;
	const size_t bytes = static_cast<size_t>(c->params.frame.npix) * sizeof(float4);
	if (async && rgba_out_host) {
		// the frame leaves on a second stream (copy engine) while the next samples are traced on the main one
		if (!c->copy_stream) { CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)); CU(cudaEventCreateWithFlags(&c->ev_resolved, cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&c->ev_copied, cudaEventDisableTiming)); }
		CU(cudaEventRecord(c->ev_resolved, c->stream));
		CU(cudaStreamWaitEvent(c->copy_stream, c->ev_resolved, 0));
		CU(cudaMemcpyAsync(rgba_out_host, c->d_fb, bytes, cudaMemcpyDeviceToHost, c->copy_stream));
		CU(cudaEventRecord(c->ev_copied, c->copy_stream));
		c->copy_pending = true;
		return B2R_OK;
	}
	if (enqueue_only) return B2R_OK;  // b2r_resolve_device: the frame stays in the device framebuffer and nobody waits
	if (rgba_out_host) CU(cudaMemcpyAsync(rgba_out_host, c->d_fb, bytes, cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	return collect_timings(c);
}

int b2r_resolve(b2r_ctx* c, float* rgba_out_host, int tonemap) { return b2r_resolve_from(c, nullptr, rgba_out_host, tonemap); }

int b2r_resolve_async(b2r_ctx* c, float* rgba_out_host, int tonemap) {
	if (!c || !rgba_out_host) return fail(B2R_ERR_ARG, "null argument");
	BucketPtrs bp{};
	for (uint32_t k = 0; k < c->cfg.buckets; k++) bp.k[k] = c->d_acc + static_cast<size_t>(k) * 3 * c->params.frame.npix;
	return resolve_with(c, bp, rgba_out_host, tonemap, true);
}
int b2r_resolve_device(b2r_ctx* c, int tonemap) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	BucketPtrs bp{};
	for (uint32_t k = 0; k < c->cfg.buckets; k++) bp.k[k] = c->d_acc + static_cast<size_t>(k) * 3 * c->params.frame.npix;
	return resolve_with(c, bp, nullptr, tonemap, false, true);
}
int b2r_frame_wait(b2r_ctx* c) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	if (c->copy_pending) { CU(cudaEventSynchronize(c->ev_copied)); c->copy_pending = false; }
	return B2R_OK;
}

int b2r_resolve_from(b2r_ctx* c, const void* dev_buckets, float* rgba_out_host, int tonemap) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	const float* base = dev_buckets ? static_cast<const float*>(dev_buckets) : c->d_acc;
	BucketPtrs bp{};
	for (uint32_t k = 0; k < c->cfg.buckets; k++) bp.k[k] = base + static_cast<size_t>(k) * 3 * c->params.frame.npix;
	return resolve_with(c, bp, rgba_out_host, tonemap);
}

int b2r_ipc_export_buckets(b2r_ctx* c, unsigned char handle_out[64]) {
	if (!c || !handle_out) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
	cudaIpcMemHandle_t h; CU(cudaIpcGetMemHandle(&h, c->d_acc));
	std::memcpy(handle_out, &h, 64);
	return B2R_OK;
}
int b2r_ipc_close(b2r_ctx* c) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	CU(sync_main(c));
	for (size_t r = 0; r < c->peer_acc.size(); r++) if (c->peer_acc[r] && r != c->my_rank) cudaIpcCloseMemHandle(c->peer_acc[r]);
	c->peer_acc.clear();
	return B2R_OK;
}
int b2r_ipc_open_peers(b2r_ctx* c, const unsigned char* peer_handles, uint32_t n_peers, uint32_t my_rank) {
	if (!c || !peer_handles || n_peers == 0 || my_rank >= n_peers) return fail(B2R_ERR_ARG, "bad peer list");
	if (c->cfg.buckets % n_peers) return fail(B2R_ERR_ARG, "bucket count must be a multiple of the number of peers");
	int rc = b2r_ipc_close(c); if (rc) return rc;
	c->peer_acc.assign(n_peers, nullptr); c->my_rank = my_rank;
	for (uint32_t r = 0; r < n_peers; r++) {
		if (r == my_rank) { c->peer_acc[r] = c->d_acc; continue; }
		cudaIpcMemHandle_t h; std::memcpy(&h, peer_handles + 64 * static_cast<size_t>(r), 64);
		cudaError_t e = cudaIpcOpenMemHandle(&c->peer_acc[r], h, cudaIpcMemLazyEnablePeerAccess);
		if (e != cudaSuccess) { c->peer_acc[r] = nullptr; b2r_ipc_close(c); return fail(B2R_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); }
	}
	return B2R_OK;
}
int b2r_resolve_peers(b2r_ctx* c, float* rgba_out_host, int tonemap) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	if (c->peer_acc.empty()) return fail(B2R_ERR_STATE, "b2r_ipc_open_peers first");
	const uint32_t G = static_cast<uint32_t>(c->peer_acc.size());
	BucketPtrs bp{};
	for (uint32_t k = 0; k < c->cfg.buckets; k++)  // bucket k lives on rank k % G (b2r_config.bucket_first/stride)
		bp.k[k] = static_cast<const float*>(c->peer_acc[k % G]) + static_cast<size_t>(k) * 3 * c->params.frame.npix;
	return resolve_with(c, bp, rgba_out_host, tonemap);
}


// ---- team mode: the multi-GPU frame without host barriers ----------------------------------------------------------------------
int b2r_team_close(b2r_ctx* c) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	CU(sync_main(c));
	if (c->copy_stream) CU(cudaStreamSynchronize(c->copy_stream));
	for (size_t r = 0; r < c->team_acc.size(); r++) if (r != c->team_rank) { if (c->team_acc[r]) cudaIpcCloseMemHandle(c->team_acc[r]); if (c->team_sync[r]) cudaIpcCloseMemHandle(c->team_sync[r]); }
	if (c->team_fb0 && c->team_rank != 0) cudaIpcCloseMemHandle(c->team_fb0);
	c->team_acc.clear(); c->team_sync.clear(); c->team_fb0 = nullptr; c->team_frame = 0; c->team_wait_done = false;
	return B2R_OK;
}
int b2r_team_export(b2r_ctx* c, unsigned char handles_out[192]) {
	if (!c || !handles_out) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	if (!c->d_team) { CU(cudaMalloc(reinterpret_cast<void**>(&c->d_team), sizeof(TeamSync))); }
	CU(cudaMemsetAsync(c->d_team, 0, sizeof(TeamSync), c->stream)); CU(sync_main(c));
	cudaIpcMemHandle_t h;
	CU(cudaIpcGetMemHandle(&h, c->d_acc)); std::memcpy(handles_out, &h, 64);
	CU(cudaIpcGetMemHandle(&h, c->d_fb)); std::memcpy(handles_out + 64, &h, 64);
	CU(cudaIpcGetMemHandle(&h, c->d_team)); std::memcpy(handles_out + 128, &h, 64);
	return B2R_OK;
}
int b2r_team_open(b2r_ctx* c, const unsigned char* all_handles, uint32_t n_ranks, uint32_t my_rank) {
	if (!c || !all_handles || n_ranks == 0 || my_rank >= n_ranks || n_ranks > static_cast<uint32_t>(kTeamMax)) return fail(B2R_ERR_ARG, "bad team (1..16 ranks)");
	if (c->cfg.buckets % n_ranks) return fail(B2R_ERR_ARG, "bucket count must be a multiple of the number of ranks");
	if (!c->d_team) return fail(B2R_ERR_STATE, "b2r_team_export first");
	int rc = b2r_team_close(c); if (rc) return rc;
	c->team_acc.assign(n_ranks, nullptr); c->team_sync.assign(n_ranks, nullptr); c->team_rank = my_rank;
	auto open = [&](void** out, const unsigned char* handle) -> int {
		cudaIpcMemHandle_t h; std::memcpy(&h, handle, 64);
		cudaError_t e = cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess);
		if (e != cudaSuccess) { *out = nullptr; return fail(B2R_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); }
		return B2R_OK;
	};
	for (uint32_t r = 0; r < n_ranks; r++) {
		const unsigned char* hs = all_handles + 192 * static_cast<size_t>(r);
		if (r == my_rank) { c->team_acc[r] = c->d_acc; c->team_sync[r] = c->d_team; continue; }
		if ((rc = open(&c->team_acc[r], hs)) || (rc = open(&c->team_sync[r], hs + 128))) { b2r_team_close(c); return rc; }
	}
	if (my_rank == 0) c->team_fb0 = c->d_fb;
	else if ((rc = open(&c->team_fb0, all_handles + 64))) { b2r_team_close(c); return rc; }
	return B2R_OK;
}
static int team_signal(b2r_ctx* c, cudaStream_t st, int field, uint32_t frame) {
	TeamPeers peers{}; const uint32_t n = static_cast<uint32_t>(c->team_sync.size());
	for (uint32_t r = 0; r < n; r++) peers.sync[r] = static_cast<TeamSync*>(c->team_sync[r]);
	k_team_signal<<<1, 32, 0, st>>>(peers, n, c->team_rank, field, frame);
	CU(cudaGetLastError()); c->launches++;
	return B2R_OK;
}
static int team_wait(b2r_ctx* c, int field, uint32_t frame) {
	k_team_wait<<<1, 32, 0, c->stream>>>(c->d_team, static_cast<uint32_t>(c->team_sync.size()), field, frame);
	CU(cudaGetLastError()); c->launches++;
	return B2R_OK;
}
// peers may still be reading this rank's buckets for the last resolved frame: anything that writes them waits (on the device) first
static int team_before_bucket_write(b2r_ctx* c) {
	if (c->team_acc.empty() || !c->team_wait_done) return B2R_OK;
	c->team_wait_done = false;
	return team_wait(c, TEAM_DONE, c->team_frame);
}
int b2r_team_resolve(b2r_ctx* c, float* rgba_out_host, int tonemap, int async) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	if (c->team_acc.empty()) return fail(B2R_ERR_STATE, "b2r_team_open first");
	int rc = ensure_device(c); if (rc) return rc;
	if (c->accumulations == 0 || c->accumulations % c->cfg.buckets) return B2R_ERR_NOT_READY;  // Renderer.hpp:437 (every rank counts every sample, so all ranks agree)
	const uint32_t G = static_cast<uint32_t>(c->team_acc.size()), f = ++c->team_frame;
	const float scale = c->params.frame.cam.exposure / static_cast<float>(c->accumulations / c->cfg.buckets);  // :439
	const bool profile = (c->cfg.flags & B2R_FLAG_NO_GRAPH) != 0;
	if ((rc = team_signal(c, c->stream, TEAM_READY, f))) return rc;   // my buckets of frame f are final (stream order: after my last accumulate)
	if ((rc = team_wait(c, TEAM_READY, f))) return rc;                // ... and so are everybody's
	if (f > 1 && (rc = team_wait(c, TEAM_COPIED, f - 1))) return rc;  // rank 0 has read frame f-1 out of its framebuffer
	BucketPtrs bp{};
	for (uint32_t k = 0; k < c->cfg.buckets; k++) bp.k[k] = static_cast<const float*>(c->team_acc[k % G]) + static_cast<size_t>(k) * 3 * c->params.frame.npix;  // bucket k lives on rank k % G
	// rank g resolves the g-th slab of 16x16 tiles (tile order) and writes it into rank 0's framebuffer
	const uint32_t n_tiles = c->params.frame.npix >> 8;
	const uint32_t t0 = static_cast<uint32_t>(static_cast<uint64_t>(n_tiles) * c->team_rank / G) << 8, t1 = static_cast<uint32_t>(static_cast<uint64_t>(n_tiles) * (c->team_rank + 1) / G) << 8;
	rc = launch(c, KK_RESOLVE, profile, [&] { k_resolve<<<c->grid_stream, kBlock, 0, c->stream>>>(c->params.frame, bp, static_cast<float4*>(c->team_fb0), scale, tonemap, t0, t1); });
	if (rc) return rc;
	if ((rc = team_signal(c, c->stream, TEAM_DONE, f))) return rc;
	c->team_wait_done = true;
	if (c->team_rank != 0) return B2R_OK;
	if ((rc = team_wait(c, TEAM_DONE, f))) return rc;  // every slab has landed in my framebuffer
	c->team_wait_done = false;
	const size_t bytes = static_cast<size_t>(c->params.frame.npix) * sizeof(float4);
	if (rgba_out_host && async) {
		if (!c->copy_stream) { CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)); CU(cudaEventCreateWithFlags(&c->ev_resolved, cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&c->ev_copied, cudaEventDisableTiming)); }
		CU(cudaEventRecord(c->ev_resolved, c->stream));
		CU(cudaStreamWaitEvent(c->copy_stream, c->ev_resolved, 0));
		CU(cudaMemcpyAsync(rgba_out_host, c->d_fb, bytes, cudaMemcpyDeviceToHost, c->copy_stream));
		if ((rc = team_signal(c, c->copy_stream, TEAM_COPIED, f))) return rc;
		CU(cudaEventRecord(c->ev_copied, c->copy_stream));
		c->copy_pending = true;
		return B2R_OK;
	}
	if (rgba_out_host) CU(cudaMemcpyAsync(rgba_out_host, c->d_fb, bytes, cudaMemcpyDeviceToHost, c->stream));
	if ((rc = team_signal(c, c->stream, TEAM_COPIED, f))) return rc;
	if (rgba_out_host) { CU(sync_main(c)); return collect_timings(c); }
	return B2R_OK;
}
int b2r_team_error(b2r_ctx* c, uint32_t* out) {
	if (!c || !out) return fail(B2R_ERR_ARG, "null argument");
	*out = 0;
	if (!c->d_team) return B2R_OK;
	int rc = ensure_device(c); if (rc) return rc;
	CU(cudaMemcpyAsync(out, &c->d_team->error, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	return B2R_OK;
}

int b2r_host_register(void* ptr, size_t bytes) {
	if (!ptr || !bytes) return fail(B2R_ERR_ARG, "null argument");
	cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterDefault);
	if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return B2R_OK; }
	if (e != cudaSuccess) return fail(B2R_ERR_CUDA, std::string("cudaHostRegister: ") + cudaGetErrorString(e));
	return B2R_OK;
}
int b2r_host_unregister(void* ptr) {
	if (!ptr) return fail(B2R_ERR_ARG, "null argument");
	cudaError_t e = cudaHostUnregister(ptr);
	if (e != cudaSuccess) { cudaGetLastError(); return fail(B2R_ERR_CUDA, std::string("cudaHostUnregister: ") + cudaGetErrorString(e)); }
	return B2R_OK;
}
int b2r_get_accumulations(b2r_ctx* c, uint32_t* out) { if (!c || !out) return fail(B2R_ERR_ARG, "null argument"); *out = c->accumulations; return B2R_OK; }
int b2r_set_accumulations(b2r_ctx* c, uint32_t acc) { if (!c) return fail(B2R_ERR_ARG, "null context"); c->accumulations = acc; drop_speculation(c); return B2R_OK; }

int b2r_read_buckets(b2r_ctx* c, float* out_host) {
	if (!c || !out_host) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	CU(cudaMemcpyAsync(out_host, c->d_acc, static_cast<size_t>(c->cfg.buckets) * 3 * c->params.frame.npix * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	return collect_timings(c);
}
int b2r_write_buckets(b2r_ctx* c, const float* in_host) {
	if (!c || !in_host) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	drop_speculation(c);
	CU(cudaMemcpyAsync(c->d_acc, in_host, static_cast<size_t>(c->cfg.buckets) * 3 * c->params.frame.npix * sizeof(float), cudaMemcpyHostToDevice, c->stream));
	CU(sync_main(c));
	return B2R_OK;
}

// ---- bucket checkpoint file (SURVEY §5 "checkpoint / resume"; the reference's only dump is the tonemapped frame, Image.cpp:71-74) --------
// Layout: 64-byte header {magic "B2RBUCK1", width, height, buckets, max_bounces, accumulations, flags that change the result, payload FNV-1a 64}
// then the [buckets][3][width*height] float32 bucket sums in tile order — exactly b2r_read_buckets' array. A progressive render resumes
// bit-identically because the RNG streams are a pure function of (sample index, pixel, bounce) (Q2-Q3).
namespace {
struct CheckpointHeader { char magic[8]; uint32_t width, height, buckets, max_bounces, accumulations, result_flags; uint64_t payload_hash; uint64_t payload_bytes; uint32_t reserved[4]; };
static_assert(sizeof(CheckpointHeader) == 64, "checkpoint header");
constexpr uint32_t kResultFlags = B2R_FLAG_NO_MIS | B2R_FLAG_REFERENCE_EXACT | B2R_FLAG_DIELECTRIC | B2R_FLAG_SKY_LIGHT | B2R_FLAG_LIGHT_TREE;  // flags that change which image is being accumulated
uint64_t fnv1a64(const void* data, size_t bytes) { const unsigned char* b = static_cast<const unsigned char*>(data); uint64_t h = 1469598103934665603ull; for (size_t i = 0; i < bytes; i++) h = (h ^ b[i]) * 1099511628211ull; return h; }
}  // namespace
int b2r_save_checkpoint(b2r_ctx* c, const char* path) {
	if (!c || !path) return fail(B2R_ERR_ARG, "null argument");
	const size_t n = static_cast<size_t>(c->cfg.buckets) * 3 * c->params.frame.npix;
	std::vector<float> host(n);
	int rc = b2r_read_buckets(c, host.data()); if (rc) return rc;
	CheckpointHeader h{}; std::memcpy(h.magic, "B2RBUCK1", 8);
	h.width = c->cfg.width; h.height = c->cfg.height; h.buckets = c->cfg.buckets; h.max_bounces = c->cfg.max_bounces; h.accumulations = c->accumulations;
	h.result_flags = c->cfg.flags & kResultFlags; h.payload_bytes = n * sizeof(float); h.payload_hash = fnv1a64(host.data(), n * sizeof(float));
	FILE* f = std::fopen(path, "wb");
	if (!f) return fail(B2R_ERR_ARG, std::string("cannot open ") + path + " for writing");
	const bool ok = std::fwrite(&h, sizeof h, 1, f) == 1 && std::fwrite(host.data(), sizeof(float), n, f) == n;
	if (std::fclose(f) != 0 || !ok) return fail(B2R_ERR_ARG, std::string("short write to ") + path);
	return B2R_OK;
}
int b2r_load_checkpoint(b2r_ctx* c, const char* path) {
	if (!c || !path) return fail(B2R_ERR_ARG, "null argument");
	FILE* f = std::fopen(path, "rb");
	if (!f) return fail(B2R_ERR_ARG, std::string("cannot open ") + path);
	CheckpointHeader h{};
	const size_t n = static_cast<size_t>(c->cfg.buckets) * 3 * c->params.frame.npix;
	std::vector<float> host(n);
	bool ok = std::fread(&h, sizeof h, 1, f) == 1 && std::memcmp(h.magic, "B2RBUCK1", 8) == 0;
	const bool same = ok && h.width == c->cfg.width && h.height == c->cfg.height && h.buckets == c->cfg.buckets && h.max_bounces == c->cfg.max_bounces &&
	                  h.result_flags == (c->cfg.flags & kResultFlags) && h.payload_bytes == n * sizeof(float);
	if (same) ok = std::fread(host.data(), sizeof(float), n, f) == n && std::fgetc(f) == EOF && fnv1a64(host.data(), n * sizeof(float)) == h.payload_hash;
	std::fclose(f);
	if (!ok) return fail(B2R_ERR_ARG, std::string(path) + ": not a bucket checkpoint, truncated, or its payload hash does not match");
	if (!same) return fail(B2R_ERR_STATE, std::string(path) + ": written for another frame size, bucket count, bounce limit (the pixel seeds depend on width and max_bounces, Q2) or MIS / reference-exact mode");
	int rc = b2r_write_buckets(c, host.data()); if (rc) return rc;
	return b2r_set_accumulations(c, h.accumulations);
}

int b2r_device_buckets(b2r_ctx* c, void** dev_ptr, size_t* bytes) {
	if (!c || !dev_ptr || !bytes) return fail(B2R_ERR_ARG, "null argument");
	*dev_ptr = c->d_acc; *bytes = static_cast<size_t>(c->cfg.buckets) * 3 * c->params.frame.npix * sizeof(float);
	return B2R_OK;
}
int b2r_device_framebuffer(b2r_ctx* c, void** dev_ptr, size_t* bytes) {
	if (!c || !dev_ptr || !bytes) return fail(B2R_ERR_ARG, "null argument");
	*dev_ptr = c->d_fb; *bytes = static_cast<size_t>(c->params.frame.npix) * sizeof(float4);
	return B2R_OK;
}

int b2r_read_counters(b2r_ctx* c, uint64_t out[10]) {
	if (!c || !out) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	unsigned long long h[ST_COUNT];
	CU(cudaMemcpyAsync(h, c->d_stats, sizeof h, cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	out[0] = h[ST_EXT]; out[1] = h[ST_SHADOW]; out[2] = h[ST_HITS]; out[3] = h[ST_TERM]; out[4] = h[ST_DROPPED]; out[5] = h[ST_SPHERE]; out[6] = h[ST_BOX];
	out[7] = c->launches; out[8] = h[ST_EVENTS]; out[9] = 0;
	return collect_timings(c);
}
int b2r_read_bounce_counts(b2r_ctx* c, uint32_t* paths_out, uint32_t* shadow_out, uint32_t n) {
	if (!c || !paths_out || !shadow_out) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	const uint32_t mb = c->cfg.max_bounces;
	const size_t block = (static_cast<size_t>(mb) + 1) * 4;
	std::vector<uint32_t> h(block * kMaxLanes);  // the last batch's counters: one block per lane (unused lanes' blocks stay zero)
	CU(cudaMemcpyAsync(h.data(), c->d_counts + static_cast<size_t>(c->counts_first) * block, kMaxLanes * c->counts_bytes, cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	for (uint32_t b = 0; b < n; b++) {
		paths_out[b] = 0u; shadow_out[b] = 0u;
		for (uint32_t j = 0; j < kMaxLanes; j++) { if (b <= mb) paths_out[b] += h[j * block + b]; if (b < mb) shadow_out[b] += h[j * block + mb + 1 + b]; }
	}
	return collect_timings(c);
}
int b2r_reset_counters(b2r_ctx* c) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	int rc = ensure_device(c); if (rc) return rc;
	CU(cudaMemsetAsync(c->d_stats, 0, ST_COUNT * sizeof(unsigned long long), c->stream));
	c->launches = 0; c->scene_epoch++;
	return B2R_OK;
}
int b2r_read_kernel_times(b2r_ctx* c, double ms_out[8], uint64_t launches_out[8], int reset) {
	if (!c || !ms_out || !launches_out) return fail(B2R_ERR_ARG, "null argument");
	int rc = ensure_device(c); if (rc) return rc;
	if ((rc = collect_timings(c))) return rc;
	for (int i = 0; i < 8; i++) { ms_out[i] = c->kernel_ms[i]; launches_out[i] = c->kernel_launches[i]; if (reset) { c->kernel_ms[i] = 0; c->kernel_launches[i] = 0; } }
	return B2R_OK;
}

int b2r_generate_rays(b2r_ctx* c, uint32_t acc, float* out_host) {
	if (!c || !out_host) return fail(B2R_ERR_ARG, "null argument");
	if (!c->have_camera) return fail(B2R_ERR_STATE, "set_camera first");
	int rc = ensure_device(c); if (rc) return rc;
	float* d = nullptr; const size_t n = static_cast<size_t>(c->params.frame.npix) * 6;
	if ((rc = dev_alloc(&d, n))) return rc;
	if (c->lens.radius > 0.0f) k_tap_generate<true><<<c->grid_stream, kBlock, 0, c->stream>>>(c->params, acc, c->lens, d);
	else k_tap_generate<false><<<c->grid_stream, kBlock, 0, c->stream>>>(c->params, acc, c->lens, d);
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess) e = cudaMemcpyAsync(out_host, d, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
	if (e == cudaSuccess) e = sync_main(c);
	cudaFree(d); c->launches++;
	if (e != cudaSuccess) return fail(B2R_ERR_CUDA, cudaGetErrorString(e));
	return B2R_OK;
}

// the leaf extents of the traversal tree must cover the finite origins of caller rays (rays[6 * i + 0..2])
static int cover_ray_origins(b2r_ctx* c, const float* rays, uint32_t n) {
	float pts[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
	for (uint32_t i = 0; i < n; i++) for (int k = 0; k < 3; k++) { const float v = rays[6 * static_cast<size_t>(i) + k]; if (v == v && fabsf(v) <= FLT_MAX) { pts[k] = fminf(pts[k], v); pts[3 + k] = fmaxf(pts[3 + k], v); } }
	return pts[0] <= pts[3] ? ensure_origin_box(c, pts, 2) : B2R_OK;
}
static int trace_common(b2r_ctx* c, const float* rays, const float* tfar_in, uint32_t n, int shadow, float* tfar_out, int32_t* prim_out, uint8_t* occ_out) {
	if (!c || !rays) return fail(B2R_ERR_ARG, "null argument");
	if (!c->have_scene) return fail(B2R_ERR_STATE, "upload_scene first");
	if (n == 0) return B2R_OK;
	int rc = ensure_device(c); if (rc) return rc;
	if (c->use_bvh && (rc = cover_ray_origins(c, rays, n))) return rc;
	c->main_reads_scene = true;  // (k_tap_trace reads the primary scene arrays on the caller's stream)
	// one grow-only device block per context, carved into the five arrays (focus picking calls this per mouse click, Application.cpp:282-298)
	const size_t n6 = (static_cast<size_t>(n) * 6 * sizeof(float) + 255) & ~static_cast<size_t>(255), n4 = (static_cast<size_t>(n) * 4 + 255) & ~static_cast<size_t>(255), n1 = (static_cast<size_t>(n) + 255) & ~static_cast<size_t>(255);
	if ((rc = dev_reserve(&c->d_trace, &c->cap_trace, n6 + 3 * n4 + n1))) return rc;
	float* d_rays = reinterpret_cast<float*>(c->d_trace); float* d_tin = reinterpret_cast<float*>(c->d_trace + n6); float* d_tout = reinterpret_cast<float*>(c->d_trace + n6 + n4);
	int32_t* d_prim = reinterpret_cast<int32_t*>(c->d_trace + n6 + 2 * n4); uint8_t* d_occ = c->d_trace + n6 + 3 * n4;
	cudaError_t e = cudaMemcpyAsync(d_rays, rays, static_cast<size_t>(n) * 6 * sizeof(float), cudaMemcpyHostToDevice, c->stream);
	if (e == cudaSuccess && shadow) e = cudaMemcpyAsync(d_tin, tfar_in, static_cast<size_t>(n) * sizeof(float), cudaMemcpyHostToDevice, c->stream);
	if (e == cudaSuccess) {
		k_tap_trace<<<c->grid_stream, kBlock, 0, c->stream>>>(c->params.scene, d_rays, d_tin, n, c->use_bvh ? 1 : 0, shadow, d_tout, d_prim, d_occ);
		e = cudaGetLastError(); c->launches++;
	}
	if (e == cudaSuccess && !shadow) { e = cudaMemcpyAsync(tfar_out, d_tout, static_cast<size_t>(n) * sizeof(float), cudaMemcpyDeviceToHost, c->stream); if (e == cudaSuccess) e = cudaMemcpyAsync(prim_out, d_prim, static_cast<size_t>(n) * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream); }
	if (e == cudaSuccess && shadow) e = cudaMemcpyAsync(occ_out, d_occ, static_cast<size_t>(n), cudaMemcpyDeviceToHost, c->stream);
	if (e == cudaSuccess) e = sync_main(c);
	if (e != cudaSuccess) return fail(B2R_ERR_CUDA, cudaGetErrorString(e));
	return B2R_OK;
}
int b2r_trace_closest(b2r_ctx* c, const float* rays_host, uint32_t n, float* tfar_out, int32_t* prim_out) {
	if (!tfar_out || !prim_out) return fail(B2R_ERR_ARG, "null argument");
	return trace_common(c, rays_host, nullptr, n, 0, tfar_out, prim_out, nullptr);
}
int b2r_trace_shadow(b2r_ctx* c, const float* rays_host, const float* tfar_host, uint32_t n, uint8_t* occluded_out) {
	if (!tfar_host || !occluded_out) return fail(B2R_ERR_ARG, "null argument");
	return trace_common(c, rays_host, tfar_host, n, 1, nullptr, nullptr, occluded_out);
}
// The per-lane kernels take caller rays in chunks of this many: a chunk is one frame of `cap` pixels (the chunk rounded up to whole
// tiles) and one sample, so ray i of a chunk has pid i.
constexpr uint32_t kTapChunk = 1u << 16;
int b2r_trace_kernel(b2r_ctx* c, int kernel, const float* rays, const float* tfar, const int32_t* origin_prim, const uint8_t* tail,
                     uint32_t n, uint32_t acc, float* tfar_out, int32_t* prim_out, uint8_t* occluded_out) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	const bool closest = kernel == B2R_TAP_CLOSEST, shadow = kernel == B2R_TAP_SHADOW, packet = kernel == B2R_TAP_PACKET;
	if (!closest && !shadow && !packet) return fail(B2R_ERR_ARG, "unknown traversal kernel");
	if ((!packet && !rays) || (shadow ? (!tfar || !origin_prim || !occluded_out) : (!tfar_out || !prim_out))) return fail(B2R_ERR_ARG, "null argument");
	if (!c->have_scene) return fail(B2R_ERR_STATE, "upload_scene first");
	if (!c->use_bvh) return fail(B2R_ERR_STATE, "the traversal kernels run on BVH contexts only");
	if (packet && !c->have_camera) return fail(B2R_ERR_STATE, "set_camera first");
	if (packet && n != c->params.frame.npix) return fail(B2R_ERR_ARG, "packet kernel: n must be width * height");
	const uint32_t n_prims = c->params.scene.n_prims;
	const bool starts = shadow || (closest && origin_prim);  // walks that start at the node holding their origin sphere (-1: the root)
	if (starts) for (uint32_t i = 0; i < n; i++) if (origin_prim[i] >= static_cast<int32_t>(n_prims)) return fail(B2R_ERR_ARG, "origin_prim out of range");
	if (n == 0) return B2R_OK;
	int rc = ensure_device(c); if (rc) return rc;
	if (!packet && (rc = cover_ray_origins(c, rays, n))) return rc;
	cudaStream_t st = c->stream;
	std::vector<uint32_t> leaf_node;  // where the walks start, as k_shade takes it for a hit on that sphere
	if (starts) { leaf_node.resize(n_prims); CU(cudaMemcpyAsync(leaf_node.data(), c->tables.leaf_node.p, n_prims * sizeof(uint32_t), cudaMemcpyDeviceToHost, st)); CU(sync_main(c)); }
	c->main_reads_scene = true;  // (the kernels read the primary scene arrays on the caller's stream)
	// one grow-only block: the queue planes, RAD, the B2R_FLAG_REFERENCE_EXACT tables, counters and batch descriptors of these launches
	// (never the context's own: its RAD may hold samples traced ahead, its queues may belong to a side in flight)
	const uint32_t chunk = packet ? n : std::min(n, kTapChunk), cap = (chunk + 255u) & ~255u;
	size_t off = 0; auto take = [&](size_t bytes) { const size_t at = off; off += (bytes + 255u) & ~static_cast<size_t>(255u); return at; };
	const size_t o_a = take(cap * sizeof(float4)), o_b = take(cap * sizeof(float4)), o_t = take(3u * cap * sizeof(float)), o_h = take(cap * sizeof(float2)),
	             o_sa = take(cap * sizeof(float4)), o_sb = take(cap * sizeof(float4)), o_sl = take(3u * cap * sizeof(float)), o_ss = take(cap * sizeof(uint32_t)),
	             o_rad = take(3u * cap * sizeof(float)), o_slot = take(cap), o_act = take(cap / 256u * sizeof(uint16_t)), o_cnt = take(16u * sizeof(uint32_t)),
	             o_stats = take(ST_COUNT * sizeof(unsigned long long)), o_batch = take((1u + kMaxLanes) * sizeof(BatchDev));
	if ((rc = dev_reserve(&c->d_tap, &c->cap_tap, off))) return rc;
	uint8_t* base = c->d_tap;
	Params p = c->params;
	p.q.A[0] = p.q.A[1] = reinterpret_cast<float4*>(base + o_a); p.q.B[0] = p.q.B[1] = reinterpret_cast<float4*>(base + o_b); p.q.T[0] = p.q.T[1] = reinterpret_cast<float*>(base + o_t);
	p.q.N[0] = p.q.N[1] = reinterpret_cast<uint32_t*>(base + o_ss);   // (a launch reads either the shadow walks' or the paths' start nodes)
	p.q.H = reinterpret_cast<float2*>(base + o_h); p.q.SA = reinterpret_cast<float4*>(base + o_sa); p.q.SB = reinterpret_cast<float4*>(base + o_sb);
	p.q.SL = reinterpret_cast<float*>(base + o_sl); p.q.SS = reinterpret_cast<uint32_t*>(base + o_ss); p.q.cap = cap;
	p.rad = reinterpret_cast<float*>(base + o_rad);
	p.ex.slot[0] = p.ex.slot[1] = base + o_slot; p.ex.act[0] = p.ex.act[1] = reinterpret_cast<uint16_t*>(base + o_act);
	uint32_t* cnt = reinterpret_cast<uint32_t*>(base + o_cnt);   // paths, shadow, work_a, work_b: four bounces each
	p.cnt.paths = cnt; p.cnt.shadow = cnt + 4; p.cnt.work_a = cnt + 8; p.cnt.work_b = cnt + 12;
	p.cnt.stats = reinterpret_cast<unsigned long long*>(base + o_stats);
	BatchDev* batch = reinterpret_cast<BatchDev*>(base + o_batch); p.batch = batch;
	const KernelSet* k = nullptr;
	if ((rc = kernels_of(c, &k))) return rc;
	std::vector<float2> h(chunk);
	if (packet) {  // one sample of the context's own frame, camera and sample index acc
		BatchArgs a; a.n = 1u; a.acc[0] = acc; a.cam = c->params.frame.cam; a.lens = c->lens;
		k_set_batch<<<1, kMaxSlots, 0, st>>>(batch, a);
		CU(cudaMemsetAsync(cnt, 0, 16u * sizeof(uint32_t), st));
		k->packet.fn<<<k->packet.grid, k->packet.block, 0, st>>>(p, 0u);
		CU(cudaGetLastError()); c->launches += 2;
		CU(cudaMemcpyAsync(h.data(), p.q.H, n * sizeof(float2), cudaMemcpyDeviceToHost, st));
		CU(sync_main(c));
		for (uint32_t i = 0; i < n; i++) { tfar_out[i] = h[i].x; std::memcpy(&prim_out[i], &h[i].y, sizeof(int32_t)); }
		return B2R_OK;
	}
	p.frame.npix = cap; p.frame.npix_magic = magic_for(cap);
	std::vector<float4> ha(chunk), hb(chunk);
	std::vector<uint32_t> hs(chunk);
	std::vector<uint8_t> hslot(chunk);
	std::vector<float> hrad(chunk);
	if (shadow) { const std::vector<float> ones(3u * static_cast<size_t>(cap), 1.0f); CU(cudaMemcpyAsync(p.q.SL, ones.data(), ones.size() * sizeof(float), cudaMemcpyHostToDevice, st)); CU(sync_main(c)); }
	else {  // with B2R_FLAG_REFERENCE_EXACT a ray takes the scalar tail when its slot >= (act & ~7) = 8: exactly the rays marked 255 below
		const std::vector<uint16_t> act(cap / 256u, static_cast<uint16_t>(8u));
		CU(cudaMemcpyAsync(p.ex.act[1], act.data(), act.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, st)); CU(sync_main(c));
	}
	for (uint32_t first = 0; first < n; first += chunk) {
		const uint32_t m = std::min(chunk, n - first);
		for (uint32_t i = 0; i < m; i++) {
			const float* r = rays + 6 * static_cast<size_t>(first + i);
			float pid; const uint32_t pid_i = i; std::memcpy(&pid, &pid_i, sizeof pid);  // slot 0, pixel i
			ha[i] = make_float4(r[0], r[1], r[2], r[3]);
			hb[i] = make_float4(r[4], r[5], shadow ? tfar[first + i] : 0.0f, pid);
			if (starts) { const int32_t o = origin_prim[first + i]; hs[i] = o < 0 ? 0u : leaf_node[o]; } else hs[i] = 0u;
			if (!shadow) hslot[i] = tail && tail[first + i] ? 255u : 0u;
		}
		uint32_t counts[16] = {0};
		if (shadow) counts[4] = m; else counts[1] = m;   // shadow rays of bounce 0 / paths entering bounce 1 (queue side 1)
		CU(cudaMemcpyAsync(cnt, counts, sizeof counts, cudaMemcpyHostToDevice, st));
		CU(cudaMemcpyAsync(shadow ? p.q.SA : p.q.A[1], ha.data(), m * sizeof(float4), cudaMemcpyHostToDevice, st));
		CU(cudaMemcpyAsync(shadow ? p.q.SB : p.q.B[1], hb.data(), m * sizeof(float4), cudaMemcpyHostToDevice, st));
		if (shadow) {
			CU(cudaMemcpyAsync(p.q.SS, hs.data(), m * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
			CU(cudaMemsetAsync(p.rad, 0, 3u * static_cast<size_t>(cap) * sizeof(float), st));
			k->shadow.fn<<<k->shadow.grid, k->shadow.block, 0, st>>>(p, 0u);
			CU(cudaGetLastError()); c->launches++;
			CU(cudaMemcpyAsync(hrad.data(), p.rad, m * sizeof(float), cudaMemcpyDeviceToHost, st));   // a lit ray adds its L = 1 to RAD
			CU(sync_main(c));
			for (uint32_t i = 0; i < m; i++) occluded_out[first + i] = hrad[i] == 0.0f ? 1u : 0u;
		} else {
			CU(cudaMemcpyAsync(p.ex.slot[1], hslot.data(), m, cudaMemcpyHostToDevice, st));
			CU(cudaMemcpyAsync(p.q.N[1], hs.data(), m * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
			k->closest.fn<<<k->closest.grid, k->closest.block, 0, st>>>(p, 1u);
			CU(cudaGetLastError()); c->launches++;
			CU(cudaMemcpyAsync(h.data(), p.q.H, m * sizeof(float2), cudaMemcpyDeviceToHost, st));
			CU(sync_main(c));
			for (uint32_t i = 0; i < m; i++) { tfar_out[first + i] = h[i].x; std::memcpy(&prim_out[first + i], &h[i].y, sizeof(int32_t)); }
		}
	}
	return B2R_OK;
}
int b2r_read_link_tables(b2r_ctx* c, uint32_t* parent_out, uint32_t* leaf_node_out) {
	if (!c || !parent_out || !leaf_node_out) return fail(B2R_ERR_ARG, "null argument");
	if (!c->have_scene) return fail(B2R_ERR_STATE, "upload_scene first");
	if (!c->use_bvh) return fail(B2R_ERR_STATE, "a brute-force context has no traversal tree");
	int rc = ensure_device(c); if (rc) return rc;
	c->main_reads_scene = true;
	CU(cudaMemcpyAsync(parent_out, c->tables.parent.p, static_cast<size_t>(c->n_wide) * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(leaf_node_out, c->tables.leaf_node.p, static_cast<size_t>(c->params.scene.n_prims) * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	return B2R_OK;
}
int b2r_read_sky_tables(b2r_ctx* c, float* marginal_out, float* conditional_out, float* pdf_out, uint32_t* cols_out, uint32_t* rows_out) {
	if (!c || !cols_out || !rows_out) return fail(B2R_ERR_ARG, "null argument");
	if (!c->have_scene) return fail(B2R_ERR_STATE, "upload_scene first");
	if (!c->sky_built) return fail(B2R_ERR_STATE, "no sky tables: B2R_FLAG_SKY_LIGHT over a sky that is not zero everywhere builds them");
	const SkyDev& k = c->params.sky;
	*cols_out = k.cols; *rows_out = k.rows;
	int rc = ensure_device(c); if (rc) return rc;
	c->main_reads_scene = true;
	if (marginal_out) CU(cudaMemcpyAsync(marginal_out, c->tables.sky_marg.p, (k.rows + 1u) * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	if (conditional_out) CU(cudaMemcpyAsync(conditional_out, c->tables.sky_cond.p, static_cast<size_t>(k.rows) * (k.cols + 1u) * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	if (pdf_out) CU(cudaMemcpyAsync(pdf_out, c->tables.sky_pdf.p, c->hdri_texels * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	return B2R_OK;
}
int b2r_read_light_tree(b2r_ctx* c, float* nodes_out, int32_t* light_prim_out, uint32_t* n_nodes_out) {
	if (!c || !n_nodes_out) return fail(B2R_ERR_ARG, "null argument");
	if (!c->have_scene) return fail(B2R_ERR_STATE, "upload_scene first");
	if (!c->lt_built || c->lt_nodes == 0u) return fail(B2R_ERR_STATE, "no light tree: B2R_FLAG_LIGHT_TREE over a scene with sphere lights builds it");
	*n_nodes_out = c->lt_nodes;
	int rc = ensure_device(c); if (rc) return rc;
	c->main_reads_scene = true;
	std::vector<int4> light(light_prim_out ? c->params.scene.n_lights : 0u);
	if (nodes_out) CU(cudaMemcpyAsync(nodes_out, c->tables.ltree_nodes.p, 2u * static_cast<size_t>(c->lt_nodes) * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
	if (light_prim_out) CU(cudaMemcpyAsync(light.data(), c->tables.ltree_light.p, light.size() * sizeof(int4), cudaMemcpyDeviceToHost, c->stream));
	CU(sync_main(c));
	for (size_t i = 0; i < light.size(); i++) light_prim_out[i] = light[i].x;
	return B2R_OK;
}
int b2r_get_origin_box(b2r_ctx* c, float out[6]) {
	if (!c || !out) return fail(B2R_ERR_ARG, "null argument");
	if (!c->obox_valid) return fail(B2R_ERR_STATE, "upload_scene first");
	for (int k = 0; k < 3; k++) { out[k] = c->obox.lo[k]; out[3 + k] = c->obox.hi[k]; }
	return B2R_OK;
}
int b2r_read_wide_nodes(b2r_ctx* c, void* out_host, uint32_t* n_wide_nodes, uint32_t* max_stack) {
	if (!c) return fail(B2R_ERR_ARG, "null context");
	if (!c->have_scene) return fail(B2R_ERR_STATE, "upload_scene first");
	if (n_wide_nodes) *n_wide_nodes = c->n_wide;
	if (max_stack) *max_stack = c->wide_host.max_stack;
	if (out_host && c->wide_refit) {  // after b2r_refit_scene the device holds the current boxes
		int rc = ensure_device(c); if (rc) return rc;
		c->main_reads_scene = true;
		CU(cudaMemcpyAsync(out_host, c->tables.wide.p, static_cast<size_t>(c->n_wide) * sizeof(WideNode), cudaMemcpyDeviceToHost, c->stream));
		CU(sync_main(c));
	} else if (out_host) std::memcpy(out_host, c->wide_host.nodes.data(), c->wide_host.nodes.size() * sizeof(WideNode));
	return B2R_OK;
}

}  // extern "C"
