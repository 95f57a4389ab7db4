#!/usr/bin/env python
"""What sampling the sky as a light buys and costs (B2R_FLAG_SKY_LIGHT), at 1920x1088, max_bounces 8, BVH pipeline:
  - scenes: BVH_test (bvh_test_scene(255)) and C3's 100k spheres (random_scene(100000), ambient 1), both under sun_hdri(2048, 1024), and
    White_Furnace (its 1x1 white sky);
  - per scene, flag off and on: frame time of SPP-sample frames enqueued back to back (one sync at the end); RMSE of an SPP-sample image
    (samples 100001..) against a REF_SPP-sample render of the same mode; efficiency = 1 / (RMSE^2 * frame time);
  - the device time of the sky's table build (k_sky_* kernels, torch.profiler) for a 2048x1024 and an 8192x4096 sun_hdri.
Prints the card name and power limit with the numbers and writes sky_workload.json into the directory given as the first argument."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpu-raytracing-experiments_b200"))
import numpy as np
import b2r, scenes

W, H, MB = 1920, 1088, 8
SPP = int(os.environ.get("SPP", "4"))
REF_SPP = int(os.environ.get("REF_SPP", "256"))
FRAMES = int(os.environ.get("FRAMES", "10"))
OUT_DIR = sys.argv[1] if len(sys.argv) > 1 else "sky_workload_out"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0]
    except Exception as e:
        return f"unknown ({e})"


def image(r, first, n):
    """mean linear radiance of samples first + 1 .. first + n, [3][npix]"""
    r.ResetAccumulator(); b2r.lib().b2r_set_accumulations(r._h, first); r.Accumulate(n); r.sync()
    return r.buckets_host().astype(np.float64).sum(axis=0) / n


def measure(sc, flags):
    r = b2r.Renderer(sc, W, H, max_bounces=MB, buckets=1, flags=flags | b2r.FLAG_FORCE_BVH)
    for _ in range(2):
        r.ResetAccumulator(); r.Accumulate(SPP); r.RenderDevice()
    r.sync()
    t0 = time.perf_counter()
    for _ in range(FRAMES):
        r.ResetAccumulator(); r.Accumulate(SPP); r.RenderDevice()
    r.sync()
    ms = (time.perf_counter() - t0) * 1e3 / FRAMES
    ref = image(r, 0, REF_SPP); img = image(r, 100000, SPP)
    r.close()
    rmse = float(np.sqrt(((img - ref) ** 2).mean()))
    return {"frame_ms": ms, "rmse": rmse, "efficiency": 1.0 / (rmse * rmse * ms * 1e-3) if rmse > 0 else None, "mean": float(ref.mean())}


def build_ms(w, h):
    import torch
    from torch.profiler import profile, ProfilerActivity
    sc = scenes.Scene(scenes.white_furnace()); sc["hdri"] = scenes.sun_hdri(w, h)
    b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_SKY_LIGHT).close()   # warm-up (module load)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_SKY_LIGHT); r.sync(); r.close()
    us = sum(e.device_time_total for e in prof.key_averages() if e.key.startswith("k_sky_") or "k_sky_" in e.key)
    return us / 1e3


def main():
    os.makedirs(OUT_DIR, exist_ok=True)
    sun = scenes.sun_hdri(2048, 1024)
    c3 = scenes.random_scene(100000); c3["ambient"] = (1.0, 1.0, 1.0); c3["hdri"] = sun
    cases = {"bvh_test_sun": scenes.bvh_test_scene(255, hdri=sun), "c3_100k_sun": c3, "white_furnace": scenes.white_furnace()}
    out = {"card": card(), "width": W, "height": H, "max_bounces": MB, "spp": SPP, "ref_spp": REF_SPP, "frames": FRAMES, "rows": []}
    print(f"card: {out['card']}  ({W}x{H}, {SPP} spp per frame, RMSE against {REF_SPP} spp of the same mode)")
    for name, sc in cases.items():
        for label, fl in (("off", 0), ("on", b2r.FLAG_SKY_LIGHT)):
            m = measure(sc, fl); m.update(scene=name, flag=label); out["rows"].append(m)
            eff = "inf (RMSE 0)" if m["efficiency"] is None else f"{m['efficiency']:.4g}"
            print(f"{name:14s} flag {label:3s}: frame {m['frame_ms']:8.2f} ms  RMSE {m['rmse']:.5g}  efficiency {eff}  mean {m['mean']:.5g}", flush=True)
    for w, h in ((2048, 1024), (8192, 4096)):
        ms = build_ms(w, h); out[f"table_build_ms_{w}x{h}"] = ms
        print(f"table build {w}x{h}: {ms:.3f} ms of device time (k_sky_*)", flush=True)
    with open(os.path.join(OUT_DIR, "sky_workload.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
