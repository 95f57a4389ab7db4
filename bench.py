#!/usr/bin/env python
"""bench.py — throughput of the hot path (Renderer::Accumulate x spp + Renderer::Render) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1|c2|c3|c4|c5] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One STEP = one frame of the workload: ResetAccumulator, Accumulate() for the workload's sample count, Render(). In the device-timed pass
(`value`) the frame is resolved into the device framebuffer and the next step is enqueued behind it without a host wait (b2r_resolve_device;
CUDA events bracket the K steps, max over ranks); in the `e2e` pass every frame is uploaded from and copied back to host memory.
Default workload = the north-star configuration, BASELINE.json configs[2] (C3): random 100k-sphere BVH scene, 1920x1080 (rendered
1920x1088, SURVEY F6), 16 spp, median-of-means with 8 buckets, max_bounces 16, light sampling + MIS. `value` is Mrays/s (extension +
shadow rays actually traced, counted on the device) with the scene resident in HBM; `e2e` is the same through the public API with host
buffers (scene upload from host, frame download to pinned host memory every step). Prints ONE JSON line on rank 0, which also carries

  * `parity_checked` / `parity`: before anything is timed the frame the N ranks produce together (buckets split over the ranks, slabs
    resolved over NVLink into rank 0's framebuffer) is compared byte for byte with the frame ONE GPU renders from the same samples, and
    with the digest committed under tests/golden/bench_digests.json when there is one; a mismatch aborts the run;
  * `strong`: the same scene at 128 spp per frame SPLIT over the ranks by bucket (strong scaling), beside the weak-scaling `value`,
    with the single-GPU time of the same frame measured in the same run (rank 0) and the resulting efficiency;
  * `e2e_dropin`: the reference's own call pattern — Accumulate() once + Render() per application frame, synchronous copy to host;
  * `c2` (N=1): the brute-force configuration BASELINE.json quotes second (default 9-sphere scene, 64 spp) as a secondary record with
    its own reference-kind CPU baseline.

--impl reference times the reference's CPU path on the host cores: the reference's own Renderer<>::Accumulate (oracle/_ref/librefrenderer.so,
compiled from /root/reference by oracle/ref_renderer_build.sh; brute force over every sphere, as shipped) on a bounded sample of the same
workload. It is the ONE place besides cpu_baseline where bench.py executes oracle/ code, as the thing being measured on the CPU.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "cpu-raytracing-experiments_b200")
sys.path[:0] = [ROOT, PKG]
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (no __pycache__ next to the modules it imports)

WORKLOADS = {
    # name: scene, width, height(internal, multiple of 16), spp, max_bounces, K
    "c1": dict(desc="C1 default 9-sphere scene 1280x720 1spp max_bounces=8 MIS K=5 (1 sample lands in bucket 1)", scene="default", w=1280, h=720, spp=5, mb=8, K=5),
    "c2": dict(desc="C2 default 9-sphere scene 1920x1080 (internal 1920x1088) 64spp median-of-means K=8 max_bounces=16 MIS brute-force", scene="default", w=1920, h=1088, spp=64, mb=16, K=8),
    "c3": dict(desc="C3 random 100k-sphere BVH scene 1920x1080 (internal 1920x1088) 16spp K=8 max_bounces=16 NEE+MIS", scene="random100000", w=1920, h=1088, spp=16, mb=16, K=8),
    "c4": dict(desc="C4 random 1M-sphere BVH scene 3840x2160 32spp K=8 max_bounces=16", scene="random1000000", w=3840, h=2160, spp=32, mb=16, K=8),
    # C5: progressive convergence run; the frame's 1024 samples are SPLIT over the ranks by bucket (strong scaling)
    "c5": dict(desc="C5 progressive 3840x2160 1024spp on the C3 100k-sphere scene, K=8 buckets split over the GPUs, max_bounces=16", scene="random100000", w=3840, h=2160, spp=1024, mb=16, K=8, strong=True),
}
STRONG_SPP = 128   # the `strong` record: this many samples per frame, split over the ranks by bucket
METRIC, UNIT = "Mrays/s", "Mrays/s"
DIGESTS = os.path.join(ROOT, "tests", "golden", "bench_digests.json")
DUMP_BYTES = 64_000_000   # --dump-outputs: payload of all .npy files of one run together


def make_scene(name):
    import scenes
    if name == "default":
        return scenes.default_scene()
    return scenes.random_scene(int(name[len("random"):]))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p)); return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every 5 ms from a thread
    (nvidia_ml_py), falling back to `nvidia-smi -lms` when NVML cannot be loaded."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu = gpu; self.sm = []; self.reasons = set(); self.mx = None; self.power = []; self.t = None; self.p = None; self.f = None; self.run = False

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            idx = self.gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.run = True

            def loop():
                while self.run:
                    try:
                        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                        r = get_reasons(h)
                        for k, b in bits.items():
                            if r & b:
                                self.reasons.add(k)
                        self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1e3)
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.t = threading.Thread(target=loop, daemon=True); self.t.start()
        except Exception:
            self.t = None
            try:
                self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
                time.sleep(0.3)
            except Exception:
                self.p = None

    def stop(self):
        if self.t is not None:
            self.run = False; self.t.join(timeout=1.0)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons), "samples": len(self.sm),
                    "power_w_max": max(self.power) if self.power else None, "source": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().strip().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------ the CPU arm
# Bounded samples. The 9-sphere scene: a few spp of the full frame. The BVH scenes: the reference brute-forces every ray against every
# sphere (USEBVH false, BVH.hpp:307), so its sample is one spp of a REDUCED frame (same scene, camera, bounce count; the frame size only
# sets how many camera rays there are) — roughly 1-5 s on the box's host cores.
CPU_REF_FRAME = {"c3": (256, 144), "c4": (128, 80), "c5": (256, 144)}
CPU_TILE_SAMPLE = {"c3": 1024, "c4": 384, "c5": 1024}


def cpu_reference_run(wl, scene, samples, first_sample=0, frame=None):
    """Times THE REFERENCE ITSELF — Renderer<>::Accumulate from /root/reference's Renderer.hpp, compiled into oracle/_ref/librefrenderer.so
    by oracle/ref_renderer_build.sh (brute force, as shipped: USEBVH false) — on all host threads. Rays are not counted by the reference;
    they are counted by the oracle on the same samples, untimed (slot-exact mode on the 9-sphere scene: bit-identical paths,
    tests/test_oracle_ref_renderer.py; its BVH mode on the large scenes, where brute-force counting would double the run: same paths up
    to grazing hits, ray counts within 1e-3)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    threads = os.cpu_count() or 1
    w, h = frame or (wl["w"], wl["h"])
    r = oracle_py.ReferenceRenderer(scene, w, h, wl["mb"])
    r.set_accumulations(first_sample)
    t0 = time.perf_counter()
    r.accumulate(samples)
    dt = time.perf_counter() - t0
    r.close()
    bvh = wl["scene"] != "default"
    o = oracle_py.Oracle(w, h, max_bounces=wl["mb"], K=5, flags=oracle_py.ORC_BVH if bvh else oracle_py.ORC_SLOT_EXACT, fast=True)
    o.set_scene(scene); o.set_accumulations(first_sample); o.reset_counters(); o.accumulate(samples, threads=threads)
    c = o.counters(); rays = c["extension_rays"] + c["shadow_rays"]; o.close()
    what = f"{samples} spp of the {w}x{h} frame" + (f" (reduced from {wl['w']}x{wl['h']}: the reference tests every ray against all {len(scene['geometry'])} spheres)" if frame else "")
    return dict(seconds=dt, rays=rays, paths=w * h * samples, threads=threads, what=what,
                mode="the reference's own Renderer::Accumulate (Renderer.hpp, g++ -O2 -mavx2 -mfma, brute force as shipped, PPL stand-in spawning its threads per parallel_for), tiles over all host threads",
                kind="reference")


def cpu_oracle_run(wl, scene, samples, fast=True, workload_name=None):
    """Times the oracle port on all host threads: `samples` x Accumulate at the workload's size (+ Render when a round completes)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle_py
    threads = os.cpu_count() or 1
    bvh = wl["scene"] != "default"
    o = oracle_py.Oracle(wl["w"], wl["h"], max_bounces=wl["mb"], K=wl["K"], flags=oracle_py.ORC_BVH if bvh else 0, fast=fast)
    o.set_scene(scene)
    o.reset_counters()
    n_tiles_all = (wl["w"] // 16) * (wl["h"] // 16)
    n_tiles = min(n_tiles_all, CPU_TILE_SAMPLE.get(workload_name, n_tiles_all)) if bvh else n_tiles_all
    t0 = time.perf_counter()
    if n_tiles < n_tiles_all:
        tiles = np.random.RandomState(1).choice(n_tiles_all, n_tiles, replace=False).astype(np.uint32)
        o.accumulate_tiles(tiles, samples, threads=threads)
    else:
        o.accumulate(samples, threads=threads); o.render()
    dt = time.perf_counter() - t0
    c = o.counters(); rays = c["extension_rays"] + c["shadow_rays"]
    o.close()
    what = f"{samples} spp of {n_tiles} of the {n_tiles_all} 16x16 tiles of the {wl['w']}x{wl['h']} frame" if n_tiles < n_tiles_all else f"{samples} spp of the {wl['w']}x{wl['h']} frame"
    return dict(seconds=dt, rays=rays, paths=n_tiles * 256 * samples, threads=threads, what=what, kind="port",
                mode="stream-BVH (BVH.hpp:320-358 restated)" if bvh else "brute force (as shipped, USEBVH false)")


def run_reference(args, wl, rank):
    """--impl reference: the CPU path on the box's host cores, one bounded sample per step."""
    if rank != 0:
        return
    scene = make_scene(wl["scene"])
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    bvh = wl["scene"] != "default"
    per_step = 1 if bvh else 4
    # the reference itself whenever it is runnable here (oracle/_ref travels with the repo; max_bounces must be one of the instantiated
    # template values); otherwise the oracle port
    use_ref = oracle_py.have_reference_renderer() and wl["mb"] in oracle_py.REF_MAX_BOUNCES and not args.cpu_port
    frame = CPU_REF_FRAME.get(args.workload) if bvh else None
    run = (lambda k: cpu_reference_run(wl, scene, per_step, first_sample=k * per_step, frame=frame)) if use_ref else (lambda k: cpu_oracle_run(wl, scene, per_step, workload_name=args.workload))
    for k in range(args.warmup):
        run(k)
    secs, rays, paths = 0.0, 0, 0
    threads = mode = what = None
    for k in range(args.steps):
        r = run(k); secs += r["seconds"]; rays += r["rays"]; paths += r["paths"]; threads, mode, what = r["threads"], r["mode"], r["what"]
    v = rays / secs / 1e6
    kind = "reference" if use_ref else "port"
    sample = f"{what} per step ({paths // args.steps} paths), {args.steps} steps; " + (mode if use_ref else f"oracle port -O3 -march=native, {mode}")
    extra = None
    if use_ref and bvh and not args.no_port_line:  # beside it: what a CPU does with the (disabled) stream-BVH branch of the reference, restated by the oracle
        p = cpu_oracle_run(wl, scene, 1, workload_name=args.workload)
        extra = {"value": p["rays"] / p["seconds"] / 1e6, "unit": UNIT, "kind": "port", "sample": f"{p['what']}; oracle port -O3 -march=native, {p['mode']} — the branch the reference compiles out (USEBVH false)"}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"]}, "paths_per_s": paths / secs,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "cpu_stream_bvh_port": extra,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": ("oracle/_ref/librefrenderer.so: the reference's Renderer.hpp and the headers it includes, compiled from /root/reference by oracle/ref_renderer_build.sh "
                 "(stand-ins for ppl.h / Image.h / glm / VCL, six token-level syntax edits; -O2, and the PPL stand-in starts its threads per parallel_for call: a few per cent against the CPU arm)") if use_ref else
                "oracle port (oracle/_ref absent, or --cpu-port)",
    }))


# ------------------------------------------------------------------------------------------------ the GPU arm
def sha(a):
    return hashlib.sha256(a.tobytes()).hexdigest()


class Bench:
    """One workload on this rank's GPU; every rank of the job builds the same object (SPMD)."""

    def __init__(self, args, name, rank, world, local, stream, dev):
        import b2r, b2r_dist
        self.b2r, self.dist_mod = b2r, b2r_dist
        self.args, self.name, self.wl, self.rank, self.world, self.local, self.stream, self.dev = args, name, WORKLOADS[name], rank, world, local, stream, dev
        wl = self.wl
        self.scene = make_scene(wl["scene"])
        self.ps = b2r.PreparedScene(self.scene, wl["w"], wl["h"])  # host BVH build + light list: scene (re)build, outside the hot path (SURVEY §3.4)
        self.K, self.spp = wl["K"], wl["spp"]
        self.base_flags = b2r.FLAG_REFERENCE_EXACT if (args.reference_exact and wl["scene"] == "default") else 0
        self.strong = bool(wl.get("strong"))
        self.step_samples = self.spp if self.strong else self.spp * world   # weak scaling: every rank renders `spp` samples of its own buckets per step
        self.r = self.renderer(sharded=True, flags=(b2r.FLAG_NO_GRAPH if args.no_graph else 0) | self.base_flags)
        self.use_team = world > 1 and args.combine == "team"
        self.use_p2p = world > 1 and args.combine == "p2p"
        if self.use_team:
            b2r_dist.open_team(self.r)
        elif self.use_p2p:
            b2r_dist.open_peers(self.r)
        self.local_buckets = b2r_dist.buckets_tensor(self.r, dev) if (world > 1 and args.combine == "nccl") else None
        self.frame_no = 0

    def renderer(self, sharded, flags=0, samples_in_flight=None):
        wl = self.wl
        shard = self.dist_mod.shard_kwargs(self.rank, self.world, self.K) if sharded else dict(bucket_first=0, bucket_stride=0)
        return self.b2r.Renderer(self.ps, wl["w"], wl["h"], max_bounces=wl["mb"], buckets=self.K, device=self.local, stream=self.stream.cuda_stream,
                                 samples_in_flight=self.args.samples_in_flight if samples_in_flight is None else samples_in_flight, flags=flags, **shard)

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def step(self, samples=None, to_host_fb=None, upload=False, async_fbs=None):
        """One frame. Multi-GPU (team mode): nothing here waits for another rank on the host — the ranks hand the frame over through flags
        in peer memory, and with async_fbs rank 0's D2H copy of frame N overlaps the tracing of frame N+1 exactly as on one GPU."""
        import torch.distributed as dist
        r = self.r
        if upload:
            r.SetScene(self.ps)  # host -> device: spheres, materials, lights, flattened BVH, camera
        r.ResetAccumulator()
        r.Accumulate(self.step_samples if samples is None else samples)
        if self.use_team:
            if async_fbs is not None:
                ok = r.RenderTeam(out=async_fbs[self.frame_no & 1], use_async=True); self.frame_no += 1
            else:
                ok = r.RenderTeam(to_host=to_host_fb is not None, out=to_host_fb)
        elif self.use_p2p:  # round-1 path, kept for comparison: rank 0 resolves everything, two host barriers per frame
            r.sync(); dist.barrier()
            ok = r.RenderPeers(to_host=to_host_fb is not None, out=to_host_fb) if self.rank == 0 else True
            dist.barrier()
        elif self.world > 1:
            r.sync()
            combined = self.dist_mod.combine_buckets(self.local_buckets)  # NCCL all-reduce of the bucket sums, then every rank resolves
            ok = r.Render(to_host=to_host_fb is not None and self.rank == 0, out=to_host_fb, dev_buckets=combined.data_ptr())
        elif async_fbs is not None:
            # progressive rendering as a user would drive it: frame N is copied out on the library's second stream into one of two pinned
            # buffers while the samples of frame N+1 are traced (b2r_resolve_async); nothing is skipped, every frame lands on the host
            ok = r.RenderAsync(async_fbs[self.frame_no & 1]); self.frame_no += 1
        elif to_host_fb is None:
            # the device-timed pass: the frame is resolved into the device framebuffer and the next frame is enqueued behind it without a host
            # wait (b2r_resolve_device) — frames are pipelined on the device exactly as the multi-GPU team path and the e2e path already are
            ok = r.RenderDevice()
        else:
            ok = r.Render(to_host=True, out=to_host_fb)
        assert ok

    def timed(self, n, **kw):
        """n steps between two barriers, timed with CUDA events on the launching stream; max over ranks."""
        import torch
        import torch.distributed as dist
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(n):
            self.step(**kw)
        if kw.get("async_fbs") is not None and (self.world == 1 or self.rank == 0):
            self.r.WaitFrame()  # the last frame has landed in host memory before the clock stops
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
        return ms

    def rays(self, cnt):
        import torch
        import torch.distributed as dist
        v = [cnt["extension_rays"] + cnt["shadow_rays"], cnt["launches"]]
        if self.world > 1:
            t = torch.tensor(v, device=self.dev, dtype=torch.float64); dist.all_reduce(t); v = [float(t[0]), float(t[1])]
        return float(v[0]), int(v[1])

    # ---- parity: the frame the job produces == the frame one GPU renders from the same samples (== the committed digest, if any)
    def parity(self, samples, tag):
        import numpy as np
        import torch
        wl = self.wl
        fb = np.zeros((wl["h"], wl["w"], 4), np.float32)
        self.step(samples=samples, to_host_fb=fb)
        self.barrier()
        out = None
        if self.rank == 0:
            # one GPU, no bucket split, a different batching (4 samples in flight, launched kernel by kernel instead of a replayed graph)
            single = self.renderer(sharded=False, flags=self.b2r.FLAG_NO_GRAPH | self.base_flags, samples_in_flight=4)
            single.Accumulate(samples); assert single.Render()
            ref = single.framebuffer.copy(); single.close()
            same = fb.tobytes() == ref.tobytes()
            key = f"{self.name}:{samples}spp" + (":exact" if self.base_flags else "")
            golden = json.load(open(DIGESTS)).get(key) if os.path.exists(DIGESTS) else None
            out = {"frame_sha256": sha(fb), "single_gpu_frame_sha256": sha(ref), "identical": bool(same), "samples_per_frame": samples, "what": tag,
                   "against": "one GPU rendering the same sample indices without the bucket split, 4 samples in flight, kernel-by-kernel launches",
                   "committed_digest": golden, "matches_committed_digest": (golden == sha(fb)) if golden else None, "digest_key": key}
            if not same:
                bad = float((fb != ref).any(axis=2).mean())
                raise SystemExit(f"bench.py: PARITY FAILURE ({tag}): the {self.world}-GPU frame differs from the single-GPU frame in {bad:.3e} of the pixels")
        self.barrier()
        if self.use_team and self.r.team_error():
            raise SystemExit("bench.py: a team hand-shake timed out")
        return out

    def close(self):
        if self.use_team:
            self.barrier(); self.r.team_close()
        self.r.close()


def device_frame(r, dev):
    """The RGBA32F frame in the renderer's device framebuffer (where b2r_resolve_device / b2r_team_resolve leave it), copied to the host."""
    import torch
    from b2r_dist import _DevArray
    r.sync()
    ptr, nbytes = r.device_framebuffer()
    return torch.as_tensor(_DevArray(ptr, nbytes // 4), device=dev).cpu().numpy().reshape(r.height, r.width, 4)


def dump_array(out_dir, name, a, budget):
    """Writes `a` as out_dir/name.npy; a frame larger than `budget` bytes is written as a fixed sample of its pixels instead (rows of the
    flattened [pixel][channel] array at ascending indices drawn with RandomState(0), so two runs sample the same pixels). Returns the bytes
    of payload written."""
    import numpy as np
    if a.nbytes > budget:
        flat = a.reshape(-1, a.shape[-1])
        keep = budget // flat[0].nbytes
        a = flat[np.sort(np.random.RandomState(0).choice(len(flat), keep, replace=False))]
    np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
    return a.nbytes


def roofline(b, kt, pc, steps, hbm_peak, peak_src, sm_max):
    """Per-kernel roofline rows from the kernel-by-kernel pass (CUDA event pair around every launch) and the device counters of the same
    steps. Algorithmic bytes / flops: DESIGN.md §5. The top-level keys describe the dominant kernel; `kernels` lists every kernel of the step."""
    wl, world, ps = b.wl, b.world, b.ps
    total_kernel_ms = sum(v[0] for v in kt.values())
    ext, shadow, hits, events, dropped = pc["extension_rays"], pc["shadow_rays"], pc["shaded_hits"], pc["radiance_events"], pc["dropped"]
    box, sph = pc.get("box_tests", 0), pc.get("sphere_tests", 0)
    npix = wl["w"] * wl["h"]
    primaries = npix * (b.step_samples // world) * steps
    fp32_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12
    rows = {}

    def row(kind, name, alg_bytes, flops=None, note=None):
        ms, n = kt[kind]
        if not n:
            return
        ach = alg_bytes / (ms / 1e3) / 1e9
        rows[name] = {"ms_per_step": ms / steps, "launches_per_step": n / steps, "avg_launch_ms": ms / n, "share_of_step": ms / total_kernel_ms if total_kernel_ms else None,
                      "algorithmic_bytes_per_launch": alg_bytes / n, "hbm_achieved_gbs": ach, "hbm_frac": ach / hbm_peak}
        if flops is not None:
            rows[name]["fp32_achieved_tflops"] = flops / (ms / 1e3) / 1e12; rows[name]["fp32_frac"] = flops / (ms / 1e3) / 1e12 / fp32_peak
        if note:
            rows[name]["note"] = note
    if kt["bounce_brute"][1]:
        n_prims = len(ps.prims)
        row("bounce_brute", "k_bounce_brute", 88.0 * (ext - primaries) + 12.0 * primaries + 24.0 * events + 12.0 * dropped,
            20.0 * n_prims * (ext + shadow) + 250.0 * hits, "44 B path record read + 44 B written per non-primary ray, 12 B radiance entry per primary path, 24 B per contribution; 20 flop per sphere test (shadow tests at their upper bound), 250 per shaded hit")
        dom = "k_bounce_brute"
    else:
        # COUNT_TESTS counters of the same steps split between the two traversal kernels in proportion to their rays (the counters are not
        # kept per kernel): 25 flop per slab test, 20 per sphere test (SURVEY §8d)
        fl = 25.0 * box + 20.0 * sph
        share_c = ext / max(ext + shadow, 1)
        row("generate", "k_generate", 56.0 * primaries, None, "44 B path record + 12 B radiance entry written per primary path")
        row("intersect_closest", "k_intersect_closest", 40.0 * ext, fl * share_c if box else None, "32 B ray read + 8 B hit record written per extension ray; nodes (128 B per visit) are L2-resident and not counted")
        row("shade", "k_shade", (8.0 + 44.0) * ext + 44.0 * (ext - primaries) + 44.0 * shadow + 24.0 * (events - 0), 250.0 * hits, "hit record + path record read per ray, path record written per continuing path, 44 B per shadow ray queued, 24 B per radiance contribution; 250 flop per shaded hit")
        row("intersect_shadow", "k_intersect_shadow", 32.0 * shadow + 12.0 * shadow, fl * (1 - share_c) if box else None, "32 B ray read per shadow ray + its 12 B light sample when unoccluded (upper bound)")
        dom = "k_intersect_closest"
    s_gpu = b.step_samples // world
    slots = b.args.samples_in_flight or min(64, max(4, (128 << 20) // npix))   # the library's default batch width (alloc_frame)
    n_batches = -(-s_gpu // slots); k_touched = min(wl["K"] // world if world > 1 else wl["K"], min(s_gpu, slots))
    row("accumulate", "k_accumulate", float(npix) * (12.0 * s_gpu + 24.0 * k_touched * n_batches) * steps, None, "12 B radiance read per (sample, pixel) + 24 B bucket read-modify-write per pixel, bucket and batch")
    row("resolve", "k_resolve", (12.0 * wl["K"] + 16.0) * npix * steps / world, None, "K bucket sums read + RGBA32F written per pixel (a rank resolves its slab)")
    d = rows[dom]
    out = {"bound": "hbm", "kernel": dom, "achieved": d["hbm_achieved_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": d["hbm_frac"], "traffic": None,
           "peak_source": peak_src, "avg_launch_ms": d["avg_launch_ms"], "launches": int(kt["bounce_brute" if dom == "k_bounce_brute" else "intersect_closest"][1]),
           "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"], "kernel_share_of_step": d["share_of_step"],
           "timing": "CUDA event pair around every launch, non-graph pass of the same steps on the launching stream",
           "note": "the traversal and brute-force kernels are bound by instruction issue and the L1/shared-memory data pipe, not by HBM: `fp32`, `issue` and `l1` say how close they are to those; `frac` is the HBM fraction the contract asks for",
           "fp32_peak_tflops": fp32_peak, "kernels": rows}
    if "fp32_achieved_tflops" in d:
        out["fp32"] = {"achieved_tflops": d["fp32_achieved_tflops"], "peak_tflops": fp32_peak, "frac": d["fp32_frac"],
                       "note": "accounting flops: 25 per slab test, 20 per sphere test (device counters, B2R_FLAG_COUNT_TESTS pass), 250 per shaded hit"}
    if box:
        out["tests_per_ray"] = {"box": box / max(ext + shadow, 1), "sphere": sph / max(ext + shadow, 1)}
    # ncu-derived figures of the same workload (static, from the committed capture profiles/r02_*): DRAM traffic per launch averaged over
    # ALL launches of the kernel in one step (the same population the algorithmic bytes per launch are averaged over), duration-weighted
    # issue-slot and L1 data-pipe utilisation, active lanes per instruction
    for fn in ("r02_traffic.json", "r01_traffic.json"):
        pth = os.path.join(ROOT, "profiles", fn)
        if not os.path.exists(pth):
            continue
        try:
            allk = json.load(open(pth)).get(b.name, {})
        except Exception:
            continue
        for kname, tr in allk.items():
            if kname in rows and world == 1:
                rows[kname]["ncu"] = {k: tr[k] for k in ("dram_bytes_per_launch", "issue_slots_busy_pct", "l1_data_pipe_pct", "active_lanes_per_instruction", "achieved_occupancy_pct", "launches") if k in tr}
                rows[kname]["traffic_over_algorithmic"] = tr["dram_bytes_per_launch"] / rows[kname]["algorithmic_bytes_per_launch"] if rows[kname]["algorithmic_bytes_per_launch"] else None
        tr = allk.get(dom)
        if tr:
            out["traffic"] = tr["dram_bytes_per_launch"]; out["traffic_source"] = tr.get("source")
            for k_src, k_dst in (("issue_slots_busy_pct", "issue"), ("l1_data_pipe_pct", "l1"), ("active_lanes_per_instruction", "active_lanes")):
                if tr.get(k_src) is not None:
                    out[k_dst] = {"value": tr[k_src], "source": "ncu, same capture as traffic"}
            break
    return out


def run_workload(args, name, rank, world, local, stream, dev, secondary=False):
    import numpy as np
    import torch
    b = Bench(args, name, rank, world, local, stream, dev)
    b2r, wl, r = b.b2r, b.wl, b.r
    warm = max(args.warmup, 3)
    steps = args.steps

    # ---- parity first: nothing is timed on a renderer whose frame is wrong
    par = b.parity(b.step_samples, f"{name}: {b.step_samples} spp per frame over {world} GPU(s)") if not args.no_parity else None

    for _ in range(warm):
        b.step()
    b.barrier()
    r.reset_counters()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms_total = b.timed(steps)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # the frame of the last timed step, before any other pass touches the framebuffer
        args.dump_left -= dump_array(args.dump_outputs, f"{name}_frame", device_frame(r, dev), args.dump_left)
    rays_total, launches = b.rays(r.counters())
    secs = ms_total / 1e3
    value = rays_total / secs / 1e6
    paths_total = wl["w"] * wl["h"] * b.step_samples * steps

    # ---- e2e: same steps through the public API with HOST buffers (scene upload + frame download each step); frames leave asynchronously
    # into two alternating pinned buffers (on one GPU: b2r_resolve_async; team mode: rank 0's copy stream), the last one is waited for
    fb_host = torch.empty((wl["h"], wl["w"], 4), dtype=torch.float32, pin_memory=True).numpy()
    fb_host2 = torch.empty((wl["h"], wl["w"], 4), dtype=torch.float32, pin_memory=True).numpy()
    e2e_kw = dict(async_fbs=[fb_host, fb_host2], upload=True) if (world == 1 or b.use_team) else dict(to_host_fb=fb_host, upload=True)
    for _ in range(2):
        b.step(**e2e_kw)
    if "async_fbs" in e2e_kw and (world == 1 or rank == 0):
        r.WaitFrame()
    r.reset_counters()
    ms_e2e = b.timed(steps, **e2e_kw)
    rays_e2e, _ = b.rays(r.counters())
    wide, _ms = r.wide_nodes()
    h2d = len(b.ps.prims) * 20 + len(b.ps.material) * 32 + max(1, len(b.ps.lights)) * 32 + wide.shape[0] * 128 + 44
    d2h = wl["w"] * wl["h"] * 16 if rank == 0 else 0
    e2e_value = rays_e2e / (ms_e2e / 1e3) / 1e6

    # ---- the drop-in's own call pattern (Application.cpp:373-382 through include/b2r_reference_binding.hpp): one Accumulate() per
    # application frame, Render() every frame — a no-op unless accumulations % K == 0, else a synchronous resolve + copy into pageable
    # host memory. N=1 only (the reference's loop knows nothing about ranks).
    dropin = None
    if world == 1 and not args.no_dropin:
        frames = 8 * wl["K"]
        page_fb = np.zeros((wl["h"], wl["w"], 4), np.float32)
        b2r.host_register(page_fb)   # as the C++ faces do with their framebuffer vector after Resize (b2r_host_register)
        def app_frames(n):
            r.ResetAccumulator()
            for _ in range(n):
                r.Accumulate(1); r.Render(out=page_fb)
        app_frames(wl["K"]); torch.cuda.synchronize(dev); r.reset_counters()
        t0 = time.perf_counter(); app_frames(frames); torch.cuda.synchronize(dev); dt = time.perf_counter() - t0
        cd = r.counters(); rd = cd["extension_rays"] + cd["shadow_rays"]
        b2r.host_unregister(page_fb)
        dropin = {"value": rd / dt / 1e6, "unit": UNIT, "ms_per_app_frame": 1e3 * dt / frames, "app_frames": frames, "resolves": frames // wl["K"],
                  "pattern": "per application frame: Accumulate() (1 sample, one wavefront batch) + Render() (resolve + synchronous D2H into the caller's frame buffer, page-locked once with b2r_host_register as the C++ faces do, when accumulations % K == 0), host wall clock",
                  "vs_batched_value": (rd / dt / 1e6) / value}

    # ---- per-kernel pass: the same steps launched kernel by kernel with an event pair around every launch (roofline), test counters on
    roof = None; kernel_ms = None
    hbm_peak, peak_src, sm_max = peaks()
    if not args.no_profile_pass:
        r.set_flags(b2r.FLAG_NO_GRAPH | b.base_flags); r.SetCamera(b.ps.camera)
        b.step(); r.sync(); r.kernel_times(reset=True); r.reset_counters()
        for _ in range(steps):
            b.step()
        r.sync()
        kt = r.kernel_times(reset=True); pc = r.counters()
        if b.r.scene is not None and wl["scene"] != "default":  # sphere / box test counts of the same steps (their own pass: counting costs time)
            r.set_flags(b2r.FLAG_NO_GRAPH | b2r.FLAG_COUNT_TESTS | b.base_flags); r.SetCamera(b.ps.camera); r.reset_counters()
            for _ in range(steps):
                b.step()
            r.sync(); cc = r.counters(); pc["box_tests"], pc["sphere_tests"] = cc["box_tests"], cc["sphere_tests"]; r.kernel_times(reset=True)
        r.set_flags(b.base_flags); r.SetCamera(b.ps.camera)
        kernel_ms = {k: {"ms": v[0], "launches": int(v[1])} for k, v in kt.items() if v[1]}
        roof = roofline(b, kt, pc, steps, hbm_peak, peak_src, sm_max)

    # ---- strong scaling beside the weak `value`: STRONG_SPP samples per frame split over the ranks by bucket
    strong = None
    if not b.strong and not secondary and not args.no_strong and wl["scene"] != "default":
        sp = b.parity(STRONG_SPP, f"{name} scene, {STRONG_SPP} spp per frame split over {world} GPU(s) by bucket") if not args.no_parity else None
        k = max(3, steps // 4)
        for _ in range(2):
            b.step(samples=STRONG_SPP)
        b.barrier(); r.reset_counters()
        ms_s = b.timed(k, samples=STRONG_SPP)
        rays_s, _ = b.rays(r.counters())
        single_ms = None
        if world > 1:
            if rank == 0:  # the same frame on ONE GPU, in the same run (the other ranks wait at the barrier)
                one = b.renderer(sharded=False, flags=b.base_flags)
                def f1():
                    one.ResetAccumulator(); one.Accumulate(STRONG_SPP); assert one.RenderDevice()
                f1(); torch.cuda.synchronize(dev)
                a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                for _ in range(k):
                    f1()
                c.record(stream); torch.cuda.synchronize(dev)
                single_ms = a.elapsed_time(c) / k; one.close()
            b.barrier()
        else:
            single_ms = ms_s / k
        strong = {"workload": f"{wl['desc'].split(' 16spp')[0]} {STRONG_SPP}spp per frame, buckets split over the GPUs (strong scaling)", "steps": k, "ms_per_step": ms_s / k,
                  "value": rays_s / (ms_s / 1e3) / 1e6, "unit": UNIT, "single_gpu_ms_per_step": single_ms,
                  "speedup_vs_one_gpu": (single_ms / (ms_s / k)) if single_ms else None, "efficiency": (single_ms / (ms_s / k) / world) if single_ms else None,
                  "parity": sp, "parity_checked": bool(sp and sp["identical"]) if rank == 0 else None}

    # ---- the same workload in B2R_FLAG_REFERENCE_EXACT mode (bit-identical to the reference's own renderer), beside the default mode's
    # number: brute-force workloads, N=1 only
    exact_line = None
    if world == 1 and not b.base_flags and wl["scene"] == "default" and not args.no_profile_pass:
        rx = b.renderer(sharded=False, flags=b2r.FLAG_REFERENCE_EXACT)
        def step_x():
            rx.ResetAccumulator(); rx.Accumulate(b.step_samples); assert rx.RenderDevice()
        for _ in range(warm):
            step_x()
        torch.cuda.synchronize(dev); rx.reset_counters()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step_x()
        e1.record(stream); torch.cuda.synchronize(dev)
        ms_x = e0.elapsed_time(e1); cx = rx.counters(); rays_x = cx["extension_rays"] + cx["shadow_rays"]
        exact_line = {"value": rays_x / (ms_x / 1e3) / 1e6, "unit": UNIT, "ms_per_step": ms_x / steps,
                      "note": "B2R_FLAG_REFERENCE_EXACT: the reference's per-tile stream order and scalar-tail sphere formula; results bit-identical to the reference's own Renderer::Accumulate/Render (tests/test_gpu_parity.py)"}
        rx.close()

    # ---- scene edit (SURVEY §8f-2; the reference rebuilds its BVH on every geometry drag, Application.cpp:508-510): every sphere of the
    # BVH workload moves by up to a quarter of its radius; b2r_refit_scene (GPU refit of the traversal tree, topology kept) beside the
    # full rebuild. Outside the timed region; N=1 only.
    edit_line = None
    if rank == 0 and world == 1 and wl["scene"] != "default" and not args.no_profile_pass and not secondary:
        rs = np.random.RandomState(5)
        geo2 = b.ps.geometry.copy(); rad = np.sqrt(geo2["radius_sq"])
        geo2["position"] += (rs.uniform(-1, 1, (len(geo2), 3)) * (0.25 * rad)[:, None]).astype(np.float32)

        def steps_ms(n=3):
            b.step(); torch.cuda.synchronize(dev)
            a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(n):
                b.step()
            c.record(stream); torch.cuda.synchronize(dev)
            return a.elapsed_time(c) / n
        r.sync(); t0 = time.perf_counter()
        r.RefitScene(geo2, want_quality=False, keep_order=True); r.sync()
        refit_ms = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        r.RefitScene(geo2, want_quality=False); r.sync()   # as the app does it: reference BVH rebuilt on the host (new leaf order), leaves re-linked
        refit_reordered_ms = (time.perf_counter() - t0) * 1e3
        q = r.RefitScene(geo2, keep_order=True)
        ms_refit = steps_ms()
        t0 = time.perf_counter()
        scene2 = dict(b.scene); scene2["geometry"] = geo2
        ps2 = b2r.PreparedScene(scene2, wl["w"], wl["h"])
        t1 = time.perf_counter()
        r.SetScene(ps2); r.sync()
        t2 = time.perf_counter()
        ms_rebuilt = steps_ms()
        edit_line = {"moved": "every sphere by up to 0.25 radius", "refit_ms": refit_ms, "refit_with_host_reference_bvh_rebuild_ms": refit_reordered_ms, "quality_ratio": q,
                     "rebuild_ms": {"reference_bvh_host": (t1 - t0) * 1e3, "upload_scene": (t2 - t1) * 1e3},
                     "ms_per_step_after_refit": ms_refit, "ms_per_step_after_rebuild": ms_rebuilt,
                     "note": "refit = match prims to geometry + pack + H2D of the spheres and lights + k_refit_level per tree level, host wall clock incl. stream sync; leaf order kept (refit_ms) or the reference BVH rebuilt on the host first, as Application.cpp:508 does"}
        # an edit that adds or removes spheres cannot keep the topology: the tree built ON THE GPU (B2R_FLAG_GPU_TREE) beside the host's SAH build
        r.set_flags(b2r.FLAG_GPU_TREE | b.base_flags); r.SetCamera(b.ps.camera); r.SetScene(ps2); r.sync()   # first use: allocations, CUB scratch
        t3 = time.perf_counter(); r.SetScene(ps2); r.sync(); t4 = time.perf_counter()
        ms_gpu_tree = steps_ms()
        edit_line["gpu_tree"] = {"upload_scene_ms": (t4 - t3) * 1e3, "ms_per_step": ms_gpu_tree,
                                 "note": "b2r_upload_scene with B2R_FLAG_GPU_TREE: pack + H2D on the host side, Hilbert keys + radix sort + implicit 4-ary links + refit passes on the device, host wall clock incl. stream sync; the balanced packed tree needs more node visits than the SAH tree (ms_per_step), so it is the instant tree after an edit, replaced by a default upload when the host build is done"}
        # the same with B2R_FLAG_GPU_SAH: the device cuts the curve order where the surface-area heuristic along the curve is smallest (k_sweep_*)
        r.set_flags(b2r.FLAG_GPU_TREE | b2r.FLAG_GPU_SAH | b.base_flags); r.SetCamera(b.ps.camera); r.SetScene(ps2); r.sync()
        t5 = time.perf_counter(); r.SetScene(ps2); r.sync(); t6 = time.perf_counter()
        ms_gpu_sweep = steps_ms()
        edit_line["gpu_sweep_tree"] = {"upload_scene_ms": (t6 - t5) * 1e3, "ms_per_step": ms_gpu_sweep, "wide_nodes": int(len(r.wide_nodes()[0])),
                                       "note": "b2r_upload_scene with B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH: as gpu_tree, but the topology is the sweep tree — per level three rounds of hand-written segmented scans (tile joins, carries, scans + cut costs in shared memory) + an open kernel over the curve order, one 4-byte read-back per level; device tree == host twin build_sweep_tree bit for bit (tests)"}
        # and with B2R_FLAG_GPU_SAH3: the three-axis sweep (x, y, z orders, the cheapest cut over all three: the host SAH tree's quality)
        r.set_flags(b2r.FLAG_GPU_TREE | b2r.FLAG_GPU_SAH3 | b.base_flags); r.SetCamera(b.ps.camera); r.SetScene(ps2); r.sync()
        t7 = time.perf_counter(); r.SetScene(ps2); r.sync(); t8 = time.perf_counter()
        ms_gpu_sweep3 = steps_ms()
        edit_line["gpu_sweep3_tree"] = {"upload_scene_ms": (t8 - t7) * 1e3, "ms_per_step": ms_gpu_sweep3, "wide_nodes": int(len(r.wide_nodes()[0])),
                                        "note": "b2r_upload_scene with B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH3: three radix-sorted orders, the scan kernels once per axis and round, the orders partitioned to match every cut; device tree == host twin build_sweep3_tree bit for bit (tests)"}
        r.set_flags(b.base_flags); r.SetCamera(b.ps.camera)
        r.SetScene(b.ps)

    # ---- CPU baseline beside it (rank 0, N=1 only): a fresh `bench.py --impl reference` process, so that its threads see the same
    # conditions as the reference arm the driver launches (inside this process, after CUDA/torch start-up, the same code ran at about half the speed)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", name, "--steps", "2", "--warmup", "1"],
                                 capture_output=True, text=True, timeout=900).stdout.strip().splitlines()[-1]
            ref = json.loads(out)
            cpu = dict(ref["cpu_baseline"]); cpu["paths_per_s"] = ref.get("paths_per_s")
            if ref.get("cpu_stream_bvh_port"):
                cpu["stream_bvh_port"] = ref["cpu_stream_bvh_port"]
        except Exception as e:  # never let the baseline leg break the GPU line
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}

    line = None
    if rank == 0:
        if b.use_team:
            part = f"sample buckets b%{world}==rank, scene+BVH replicated; team mode: every rank resolves its slab of tiles reading the bucket sums from their owners over NVLink (CUDA IPC) and stores it into rank 0's framebuffer; hand-shakes are release/acquire flags in peer memory (no host barrier per frame)"
        elif b.use_p2p:
            part = f"sample buckets b%{world}==rank; resolve kernel on rank 0 reads peer bucket arrays over NVLink (CUDA IPC), 2 host barriers per frame"
        elif world > 1:
            part = f"sample buckets b%{world}==rank; one NCCL all-reduce of bucket sums per frame"
        else:
            part = "single GPU"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": ms_total / steps,
            "higher_is_better": True, "scaling": "strong" if b.strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"] + (" [B2R_FLAG_REFERENCE_EXACT: reference's stream order and scalar-tail formula]" if b.base_flags else ""), "samples_per_step_per_gpu": b.step_samples // world, "samples_in_flight": args.samples_in_flight,
                       "partition": part,
                       "l2": "no flush needed: each step streams >1 GB of path-queue records (>> 126 MB L2); RNG-unique samples every step",
                       "frames": "enqueued back to back: every step resets, traces, folds and resolves its frame into the device framebuffer; no host wait inside the timed region, so the device pipelines consecutive frames (the e2e figure copies every frame to the host)"},
            "paths_per_s": paths_total / secs, "rays_per_step": rays_total / steps,
            "parity_checked": bool(par and par["identical"]), "parity": par,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e / steps,
                    "includes": "upload_scene (pack + 128-B BVH flatten on host, H2D), set_camera, reset, Accumulate x spp, Render, D2H of the RGBA32F frame into pinned memory"
                                + ("; frames leave asynchronously (copy of frame N overlaps the tracing of frame N+1, two pinned buffers, last frame waited for inside the timed region)" if "async_fbs" in e2e_kw else "")},
            "e2e_dropin": dropin, "strong": strong,
            "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu, "kernel_ms": kernel_ms,
        }
        if exact_line:
            line["reference_exact_mode"] = exact_line
        if edit_line:
            line["scene_edit"] = edit_line
    b.close()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1); ap.add_argument("--steps", type=int, default=20); ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"]); ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true"); ap.add_argument("--no-profile-pass", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the frame-hash check (ncu runs only; a reported number always carries it)")
    ap.add_argument("--no-strong", action="store_true"); ap.add_argument("--no-dropin", action="store_true"); ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--cpu-port", action="store_true", help="--impl reference: time the oracle port instead of the reference itself")
    ap.add_argument("--no-port-line", action="store_true")
    ap.add_argument("--samples-in-flight", type=int, default=0, help="0 = library default (auto)")
    ap.add_argument("--no-graph", action="store_true", help="launch kernel by kernel (for ncu); never used for a reported number")
    ap.add_argument("--reference-exact", action="store_true", help="brute-force workloads: B2R_FLAG_REFERENCE_EXACT (bit-identical to the reference's own renderer; one extra ranking kernel per bounce)")
    ap.add_argument("--combine", default="team", choices=["team", "p2p", "nccl"], help="multi-GPU frame combine: team = sliced resolve over NVLink with device-side hand-shakes (default); p2p = rank 0 resolves, host barriers (round 1); nccl = all-reduce then resolve")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps of each workload, write the RGBA32F frame of its last step as DIR/<workload>_frame.npy "
                    "(float32 [height][width][4]; a frame that does not fit the 64 MB left for the run is written as a fixed sample of its pixels, [pixels][4]: "
                    "the rows of the flattened [height*width][4] frame at the indices np.sort(np.random.RandomState(0).choice(height*width, pixels, replace=False)))")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "ours":
            ap.error("--dump-outputs writes the GPU path's frames: --impl ours only")
        os.makedirs(args.dump_outputs, exist_ok=True)
    args.dump_left = DUMP_BYTES - 4096   # (4 KB for the .npy headers)
    args.warmup = max(args.warmup, 0)
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, wl, rank); return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    if rank == 0:
        entry.build()
    if world > 1:
        torch.cuda.set_device(local)
        # NCCL prints its version banner to stdout when the first communicator is created: file descriptor 1 points at /dev/null until
        # that has happened, so that rank 0's stdout carries ONE line
        sys.stdout.flush(); keep = os.dup(1); null = os.open(os.devnull, os.O_WRONLY); os.dup2(null, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
            dist.barrier()
            t = torch.zeros(1, device=f"cuda:{local}"); dist.all_reduce(t); torch.cuda.synchronize()
        finally:
            sys.stdout.flush(); os.dup2(keep, 1); os.close(keep); os.close(null)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libb2r has no CPU fallback")
    dev = torch.device(f"cuda:{local}"); torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)  # a real (non-default) stream: the library launches on it and the timing events are recorded on it
    torch.cuda.set_stream(stream)

    line = run_workload(args, args.workload, rank, world, local, stream, dev)
    # secondary record: BASELINE.json configs[1] (C2, the brute-force configuration the reference itself can run at full size), N=1
    if world == 1 and args.workload == "c3" and not args.no_secondary and not args.no_graph:
        c2 = run_workload(args, "c2", rank, world, local, stream, dev, secondary=True)
        if rank == 0:
            line["c2"] = {k: c2[k] for k in ("value", "unit", "ms_per_step", "config", "paths_per_s", "parity_checked", "parity", "e2e", "e2e_dropin", "roofline", "cpu_baseline", "kernel_ms", "reference_exact_mode") if k in c2}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
