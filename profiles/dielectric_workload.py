#!/usr/bin/env python
"""What glass costs (B2R_FLAG_DIELECTRIC):
  - C3's scene (random_scene(100000), 1920x1088, 16 spp, K = 8, max_bounces 16, BVH pipeline) with 0, 1 and 2 of its 8 materials made glass
    (IOR 1.5, transmission 0.95), all with the flag: frame time with frames enqueued back to back (RenderDevice, one sync at the end), and the
    paths entering and shadow rays queued at each bounce of the last wavefront batch (Renderer.bounce_counts());
  - C3 without the flag (the existing kernels), the reference point for the 0-glass row;
  - the default scene at C2's size (1920x1088, 64 spp, K = 8, max_bounces 16, brute force) without and with the flag (its ball and gem glass).
Writes the default scene rendered with the flag as default_dielectric.hdr (b2r_write_hdr, linear RGBA32F). Prints the card name and power
limit with the numbers and writes dielectric_workload.json into the directory given as the first argument (default: ./dielectric_workload_out)."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpu-raytracing-experiments_b200"))
import numpy as np
import b2r, scenes

W, H, MB, K = 1920, 1088, 16, 8
FRAMES = int(os.environ.get("FRAMES", "10"))
OUT_DIR = sys.argv[1] if len(sys.argv) > 1 else "dielectric_workload_out"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0]
    except Exception as e:
        return f"unknown ({e})"


def glass(sc, mats):
    sc = scenes.Scene(sc); m = np.ascontiguousarray(sc["material"]).copy()
    for k in mats:
        m[k]["transmission"] = np.float32(0.95); m[k]["IOR_minus_one"] = np.float32(0.5)
    sc["material"] = m
    return sc


def measure(sc, spp, flags, frames=FRAMES):
    r = b2r.Renderer(sc, W, H, max_bounces=MB, buckets=K, flags=flags)
    for _ in range(2):   # warm-up frames (graph capture, clocks)
        r.ResetAccumulator(); r.Accumulate(spp); r.RenderDevice()
    r.sync()
    t0 = time.perf_counter()
    for _ in range(frames):
        r.ResetAccumulator(); r.Accumulate(spp); r.RenderDevice()
    r.sync(); ms = (time.perf_counter() - t0) * 1e3 / frames
    paths, shadow = r.bounce_counts()
    assert r.Render(); fb = r.framebuffer.copy(); r.close()
    return ms, paths.tolist(), shadow.tolist(), fb


def main():
    os.makedirs(OUT_DIR, exist_ok=True)
    info = card()
    print(f"card: {info}; {W}x{H} K={K} mb={MB}, {FRAMES} frames per row")
    rows = []
    c3 = scenes.random_scene(100000)
    for name, sc, flags in [("c3_no_flag", c3, 0), ("c3_glass0", c3, b2r.FLAG_DIELECTRIC), ("c3_glass1", glass(c3, [1]), b2r.FLAG_DIELECTRIC),
                            ("c3_glass2", glass(c3, [1, 4]), b2r.FLAG_DIELECTRIC), ("c3_no_flag_again", c3, 0)]:
        ms, paths, shadow, _ = measure(sc, 16, flags)
        row = dict(name=name, spp=16, frame_ms=ms, paths=paths, shadow=shadow); rows.append(row); print(json.dumps(row))
    d = scenes.default_scene()
    for name, flags in [("c2_no_flag", b2r.FLAG_FORCE_BRUTE), ("c2_dielectric", b2r.FLAG_FORCE_BRUTE | b2r.FLAG_DIELECTRIC), ("c2_no_flag_again", b2r.FLAG_FORCE_BRUTE)]:
        ms, paths, shadow, fb = measure(d, 64, flags)
        row = dict(name=name, spp=64, frame_ms=ms, paths=paths, shadow=shadow); rows.append(row); print(json.dumps(row))
        if name == "c2_dielectric":
            b2r.write_hdr(os.path.join(OUT_DIR, "default_dielectric.hdr"), fb)
        if name == "c2_no_flag":
            b2r.write_hdr(os.path.join(OUT_DIR, "default_opaque.hdr"), fb)
    json.dump(dict(card=info, frames=FRAMES, rows=rows, lib=b2r.LIB_PATH), open(os.path.join(OUT_DIR, "dielectric_workload.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
