#!/usr/bin/env python
"""What picking sphere lights from the light tree buys and costs (B2R_FLAG_LIGHT_TREE), BVH pipeline, max_bounces 16, K = 8 buckets:
  - scenes: C3 (random_scene(100000): 100 emitters) at 1920x1088 and C4 (random_scene(1000000): 1000 emitters) at 1920x1088 (C4's 3840x2160
    is not needed for a ratio);
  - per scene, flag off and on, alternating in one run (ROUNDS rounds): the frame time of SPP-sample frames (K | SPP) enqueued back to back;
  - per-pixel variance per sample across the median-of-means buckets of one SPP-sample frame: var over the K bucket means of each pixel
    (channel mean) times SPP / K, averaged over the pixels, and relative to the squared frame mean (the two modes have different expectations:
    without the flag quirks Q9 and Q10 bias the sphere lights' estimate);
  - efficiency = 1 / (relative variance per sample x frame time).
Prints the card name and power limit with the numbers and writes light_tree_workload.json into the directory given as the first argument."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpu-raytracing-experiments_b200"))
import numpy as np
import b2r, scenes

W, H, MB, K = 1920, 1088, 16, 8
SPP = int(os.environ.get("SPP", "16"))
ROUNDS = int(os.environ.get("ROUNDS", "3"))
FRAMES = int(os.environ.get("FRAMES", "4"))
OUT_DIR = sys.argv[1] if len(sys.argv) > 1 else "light_tree_workload_out"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0]
    except Exception as e:
        return f"unknown ({e})"


def frame_ms(r):
    r.sync(); t0 = time.perf_counter()
    for _ in range(FRAMES):
        r.ResetAccumulator(); r.Accumulate(SPP); r.RenderDevice()
    r.sync()
    return (time.perf_counter() - t0) * 1e3 / FRAMES


def variance(r):
    r.ResetAccumulator(); r.Accumulate(SPP); r.sync()
    b = r.buckets_host().astype(np.float64).mean(axis=1) / (SPP // K)   # [K][npix]: each bucket's mean per sample
    var = float(b.var(axis=0, ddof=1).mean()) * (SPP // K)              # per sample
    mean = float(b.mean())
    return var, mean


def main():
    os.makedirs(OUT_DIR, exist_ok=True)
    out = {"card": card(), "width": W, "height": H, "max_bounces": MB, "buckets": K, "spp": SPP, "rounds": ROUNDS, "frames": FRAMES, "rows": []}
    print(f"card: {out['card']}  ({W}x{H}, {SPP} spp per frame in {K} buckets, max_bounces {MB}, BVH pipeline)", flush=True)
    for name, n in (("C3", 100000), ("C4", 1000000)):
        sc = scenes.random_scene(n)
        rs = {fl: b2r.Renderer(sc, W, H, max_bounces=MB, buckets=K, flags=fl | b2r.FLAG_FORCE_BVH) for fl in (0, b2r.FLAG_LIGHT_TREE)}
        for r in rs.values():
            r.ResetAccumulator(); r.Accumulate(SPP); r.RenderDevice(); r.sync()   # warm-up: graphs captured, modules loaded
        times = {fl: [] for fl in rs}
        for _ in range(ROUNDS):
            for fl, r in rs.items(): times[fl].append(frame_ms(r))
        row = {"scene": name, "spheres": n}
        for fl, r in rs.items():
            var, mean = variance(r); ms = float(np.median(times[fl]))
            rel = var / (mean * mean)
            key = "on" if fl else "off"
            row[key] = {"frame_ms": ms, "frame_ms_all": times[fl], "var_per_sample": var, "mean": mean, "rel_var_per_sample": rel, "efficiency": 1.0 / (rel * ms * 1e-3)}
            r.close()
        row["frame_time_ratio"] = row["on"]["frame_ms"] / row["off"]["frame_ms"]
        row["rel_var_ratio"] = row["on"]["rel_var_per_sample"] / row["off"]["rel_var_per_sample"]
        row["var_ratio"] = row["on"]["var_per_sample"] / row["off"]["var_per_sample"]
        row["efficiency_ratio"] = row["on"]["efficiency"] / row["off"]["efficiency"]
        out["rows"].append(row)
        for key in ("off", "on"):
            m = row[key]
            print(f"{name} flag {key:3s}: frame {m['frame_ms']:8.2f} ms  mean {m['mean']:.5g}  var/sample {m['var_per_sample']:.5g}  rel var/sample {m['rel_var_per_sample']:.5g}"
                  f"  efficiency {m['efficiency']:.5g}", flush=True)
        print(f"{name} on/off: frame time {row['frame_time_ratio']:.3f}x  variance {row['var_ratio']:.3f}x  relative variance {row['rel_var_ratio']:.3f}x"
              f"  efficiency {row['efficiency_ratio']:.3f}x", flush=True)
    with open(os.path.join(OUT_DIR, "light_tree_workload.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
