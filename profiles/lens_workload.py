#!/usr/bin/env python
"""What a thin lens costs (b2r_set_lens): C3's scene (random_scene(100000), 1920x1088, 16 spp, K = 8, max_bounces 16) with R = 0 (the
pinhole) and three lens radii focused at the scene centre, from a few pixels of blur to a large fraction of the scene. For each:
  - frame time: 16 samples per frame, frames enqueued back to back (RenderDevice), one sync at the end;
  - bounce-0 time of the packet kernel: kernel_times() under FLAG_NO_GRAPH (the intersect_closest launches of bounce 0 of every batch);
  - box tests (about 4 per node visit) and sphere tests per primary ray: FLAG_COUNT_TESTS counters of a max_bounces = 1 frame, where the
    packet kernel is the only traversal;
  - the lens with B2R_NO_PACKET (k_generate + the per-lane walk at bounce 0) against the packet kernel.
Prints the card name and power limit with the numbers and writes lens_workload.json into the directory given as the first argument
(default: ./lens_workload_out)."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpu-raytracing-experiments_b200"))
import numpy as np
import b2r, scenes

W, H, SPP, MB, K = 1920, 1088, 16, 16, 8
FRAMES = int(os.environ.get("FRAMES", "20"))
REPS = int(os.environ.get("REPS", "3"))
OUT = os.path.join(sys.argv[1] if len(sys.argv) > 1 else "lens_workload_out", "lens_workload.json")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0]
    except Exception as e:
        return f"unknown ({e})"


def frame_ms(ps, lens, no_packet=False):
    if no_packet: os.environ["B2R_NO_PACKET"] = "1"
    else: os.environ.pop("B2R_NO_PACKET", None)
    r = b2r.Renderer(ps, W, H, max_bounces=MB, buckets=K)
    r.SetLens(*lens)
    for _ in range(3):   # warm-up frames (graph capture, clocks)
        r.ResetAccumulator(); r.Accumulate(SPP); r.RenderDevice()
    r.sync()
    t0 = time.perf_counter()
    for _ in range(FRAMES):
        r.ResetAccumulator(); r.Accumulate(SPP); r.RenderDevice()
    r.sync(); t = (time.perf_counter() - t0) * 1e3 / FRAMES
    r.close(); os.environ.pop("B2R_NO_PACKET", None)
    return t


def bounce0_ms(ps, lens, no_packet=False):
    """bounce-0 traversal time per frame: FLAG_NO_GRAPH times every launch; the first intersect_closest launch of a batch is bounce 0"""
    if no_packet: os.environ["B2R_NO_PACKET"] = "1"
    r = b2r.Renderer(ps, W, H, max_bounces=1, buckets=K, flags=b2r.FLAG_NO_GRAPH)   # max_bounces 1: every intersect_closest launch is bounce 0
    r.SetLens(*lens); r.Accumulate(SPP); r.sync(); r.kernel_times(reset=True)
    for _ in range(REPS):
        r.ResetAccumulator(); r.Accumulate(SPP)
    r.sync()
    kt = r.kernel_times(reset=True); r.close(); os.environ.pop("B2R_NO_PACKET", None)
    return (kt["intersect_closest"][0] + (kt["generate"][0] if no_packet else 0.0)) / REPS, kt["intersect_closest"][1] // REPS


def counts(ps, lens):
    r = b2r.Renderer(ps, W, H, max_bounces=1, buckets=K, flags=b2r.FLAG_COUNT_TESTS)
    r.SetLens(*lens); r.reset_counters()
    r.Accumulate(SPP); r.sync()
    c = r.counters(); r.close(); n = W * H * SPP
    return c["box_tests"] / n, c["sphere_tests"] / n


def main():
    sc = scenes.random_scene(100000); ps = b2r.PreparedScene(sc, W, H)
    g = sc["geometry"]; centre = g["position"].astype(np.float64).mean(0)
    eye = np.asarray(sc["camera"]["eye"], np.float64); F = float(np.linalg.norm(centre - eye))
    lo, hi = g["position"].min(0), g["position"].max(0); extent = float((hi - lo).max())
    cam = ps.camera; z = abs(float(cam[9]))
    # a lens of radius R blurs a point at depth d by 2 R |z| |d - F| / (d F) pixels; the radii below give about 4 pixels of blur at depth 2F,
    # then 0.5 % and 5 % of the scene's extent
    radii = [0.0, 4.0 * F / z, 0.005 * extent, 0.05 * extent]
    info = card()
    print(f"card: {info}; C3 {W}x{H} {SPP} spp K={K} mb={MB}; focus distance {F:.2f} (scene centre), extent {extent:.1f}, |z| {z:.1f} px")
    rows = []
    for R in radii + [0.0]:   # the pinhole again at the end: the spread of the same measurement
        lens = (R, F)
        row = dict(radius=R, focus=F, blur_px_at_2F=R * z / F, frame_ms=frame_ms(ps, lens))
        row["bounce0_packet_ms"], row["bounce0_launches"] = bounce0_ms(ps, lens)
        row["box_tests_per_primary"], row["sphere_tests_per_primary"] = counts(ps, lens)
        if R > 0.0:
            row["frame_ms_no_packet"] = frame_ms(ps, lens, no_packet=True)
            row["bounce0_no_packet_ms"], _ = bounce0_ms(ps, lens, no_packet=True)
        rows.append(row)
        print(json.dumps(row))
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    json.dump(dict(card=info, workload=f"c3 {W}x{H} {SPP}spp K={K} mb={MB}", frames=FRAMES, rows=rows, lib=b2r.LIB_PATH), open(OUT, "w"), indent=1)


if __name__ == "__main__":
    main()
