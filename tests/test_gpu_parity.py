"""GPU parity tests (-m gpu): the sm_100a kernels, called through the C ABI (libb2r.so), against the CPU oracle on the same
scene, camera, seeds and bounce count; against committed golden fixtures; and, at BASELINE.json's full sizes, through
size-independent properties (BVH traversal == brute force on the GPU itself, oracle spot-check tiles, sample-range additivity).

Tolerances (north_star): BVH node and leaf order bit-exact; per-sample pixel radiance within 1e-4 relative with the fraction of
divergent pixels reported (asserted small); converged image RMSE < 1e-3. The brute-force pipeline is in fact bit-exact.
"""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

import b2r
import oracle_py
import scenes

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
REL_TOL = 1e-4


def divergent_fraction(a, b):
    """fraction of pixels whose radiance differs by more than 1e-4 relative in any channel/bucket"""
    rel = np.abs(a - b) / np.maximum(np.abs(b), 1e-6)
    return float((rel > REL_TOL).any(axis=tuple(range(a.ndim - 1))).mean())


def oracle_for(sc, w, h, mb, K, flags=0):
    o = oracle_py.Oracle(w, h, max_bounces=mb, K=K, flags=flags); o.set_scene(sc); return o


# ------------------------------------------------------------------------------------------------ stage-level parity
def test_camera_rays_bit_exact():
    sc = scenes.default_scene()
    for (w, h, mb, acc) in [(1280, 720, 8, 1), (1920, 1088, 16, 64), (320, 192, 16, 1024)]:
        r = b2r.Renderer(sc, w, h, max_bounces=mb)
        o = oracle_for(sc, w, h, mb, 5)
        assert r.generate_rays(acc).tobytes() == o.generate_rays(acc).tobytes()
        r.close()


@pytest.mark.parametrize("n,flags", [(9, 0), (300, b2r.FLAG_FORCE_BRUTE), (300, b2r.FLAG_FORCE_BVH), (20000, b2r.FLAG_FORCE_BVH)])
def test_traverse_api_vs_bruteforce_oracle(n, flags):
    """BoundingVolumeHierarchy::Traverse / Traverse_shadow on caller rays (Application.cpp:282-298)."""
    sc = scenes.default_scene() if n == 9 else scenes.random_scene(n, light_every=50)
    r = b2r.Renderer(sc, 64, 64, flags=flags); o = oracle_for(sc, 64, 64, 16, 1)
    rs = np.random.RandomState(n)
    m = 20000 if n <= 300 else 3000
    span = 3.0 if n == 9 else 150.0
    rays = np.zeros((m, 6), np.float32); rays[:, :3] = rs.uniform(-span, span, (m, 3)); d = rs.randn(m, 3); rays[:, 3:] = d / np.linalg.norm(d, axis=1, keepdims=True)
    t, p = r.trace_closest(rays); to, po = o.trace_closest(rays)
    mismatch = float((p != po).mean())
    print(f"closest-hit prim mismatch fraction n={n} flags={flags}: {mismatch:.2e}")
    assert mismatch == 0.0 and t.tobytes() == to.tobytes()   # the BVH's hit decisions equal brute force exactly (DESIGN §2)
    tf = rs.uniform(1.0, 2 * span, m).astype(np.float32)
    occ = r.trace_shadow(rays, tf); occ_o = o.trace_shadow(rays, tf)
    assert np.array_equal(occ, occ_o)
    r.close()


# ------------------------------------------------------------------------------------------------ per-sample radiance
def test_c1_default_scene_720p_one_sample():
    """BASELINE configs[0]: default scene, 1280x720, 1 spp, max_bounces 8 — the reference's own CPU-runnable case."""
    sc = scenes.default_scene()
    r = b2r.Renderer(sc, 1280, 720, max_bounces=8, buckets=5); r.Accumulate(1)
    o = oracle_for(sc, 1280, 720, 8, 5); o.accumulate(1)
    g, ref = r.buckets_host(), o.buckets()
    frac = divergent_fraction(g, ref)
    print(f"C1 divergent pixel fraction {frac:.3e}; bit-exact: {g.tobytes() == ref.tobytes()}")
    assert frac == 0.0 and g.tobytes() == ref.tobytes()
    gc, oc = r.counters(), o.counters()
    assert gc["extension_rays"] == oc["extension_rays"] and gc["shaded_hits"] == oc["shaded_hits"]
    assert gc["terminated"] == oc["terminated"] and gc["dropped"] == oc["dropped"] and gc["shadow_rays"] <= oc["shadow_rays"]
    r.close()


def test_golden_fixture_without_oracle():
    g = json.load(open(os.path.join(G, "oracle_frames.json")))
    sc = scenes.default_scene()
    r = b2r.Renderer(sc, 320, 192, max_bounces=8, buckets=5); r.Accumulate(5)
    assert hashlib.sha256(r.buckets_host().tobytes()).hexdigest() == g["default_320x192_mb8_K5_acc5"]["sha256_buckets"]
    assert r.Render()
    assert hashlib.sha256(r.framebuffer.tobytes()).hexdigest() == g["default_320x192_render_sha256"]
    r2 = b2r.Renderer(sc, 160, 96, max_bounces=16, buckets=1); r2.accumulations = 63; r2.Accumulate(1)
    assert hashlib.sha256(r2.buckets_host().tobytes()).hexdigest() == g["default_160x96_mb16_K1_acc64"]["sha256_buckets"]
    sc3 = scenes.random_scene(2000, light_every=50)
    r3 = b2r.Renderer(sc3, 160, 96, max_bounces=8, buckets=1, flags=b2r.FLAG_FORCE_BRUTE); r3.Accumulate(1)
    assert hashlib.sha256(r3.buckets_host().tobytes()).hexdigest() == g["random2000_160x96_mb8_K1_acc1"]["sha256_buckets"]
    for x in (r, r2, r3): x.close()


@pytest.mark.parametrize("K,n", [(5, 65), (8, 64)])
def test_c2_median_of_means_resolve(K, n):
    """BASELINE configs[1] semantics at reduced size: n samples into K buckets, median-of-means + ACES (Renderer.hpp:436-478).
    K=5/65 is the reference-exact variant (Q21), K=8/64 this repo's definition of '8 buckets'."""
    sc = scenes.default_scene()
    w, h = 480, 272
    r = b2r.Renderer(sc, w, h, max_bounces=16, buckets=K); o = oracle_for(sc, w, h, 16, K)
    for step in (n - K, K):  # Render() is a no-op unless accumulations % K == 0 (Renderer.hpp:437)
        r.Accumulate(step); o.accumulate(step)
    assert r.accumulations == n and r.Render()
    rc, ref = o.render(); assert rc == 0
    assert divergent_fraction(r.buckets_host(), o.buckets()) == 0.0
    rmse = float(np.sqrt(np.mean((r.framebuffer - ref) ** 2)))
    print(f"K={K} converged tonemapped RMSE {rmse:.3e}; framebuffer bit-exact: {r.framebuffer.tobytes() == ref.tobytes()}")
    assert rmse < 1e-3 and np.all(r.framebuffer[..., 3] == 1.0)
    lin = np.zeros_like(r.framebuffer); assert r.Render(tonemap=False, out=lin)
    assert float(np.sqrt(np.mean((lin - o.render(tonemap=False)[1]) ** 2))) < 1e-3
    r.Accumulate(1); before = r.framebuffer.copy(); assert not r.Render() and np.array_equal(before, r.framebuffer)
    r.close()


@pytest.mark.parametrize("n,w,h,mb,tree", [(600, 192, 112, 6, 0), (5000, 160, 96, 8, 0), (5000, 160, 96, 8, b2r.FLAG_REFERENCE_TREE)])
def test_bvh_pipeline_vs_bruteforce_oracle(n, w, h, mb, tree):
    """The flattened-BVH wavefront (intersect -> shade -> shadow kernels) against the brute-force oracle (the semantics the
    reference ships, USEBVH false): bit-identical, the tree being conservative against the float sphere tests (DESIGN §2)."""
    sc = scenes.random_scene(n, light_every=40)
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=2, flags=b2r.FLAG_FORCE_BVH | tree); r.Accumulate(4)
    o = oracle_for(sc, w, h, mb, 2); o.accumulate(4)
    frac = divergent_fraction(r.buckets_host(), o.buckets())
    print(f"BVH pipeline n={n} tree={tree}: divergent pixel fraction {frac:.3e}")
    assert r.buckets_host().tobytes() == o.buckets().tobytes()
    gc, oc = r.counters(), o.counters()
    assert gc["extension_rays"] == oc["extension_rays"]
    r.close()


def test_deep_traversal_stack_nested_spheres():
    """Every box of this scene overlaps every other (4096 large spheres whose centres sit within two units), so each node visit
    hits all its children and the per-lane traversal stack grows by three per level: the shared-memory part of the stack
    (16 entries) overflows on essentially every ray and the bulk evict / refill path of the persistent kernels runs. Results
    must still equal brute force."""
    sc = scenes.random_scene(4096, light_every=64)
    rs = np.random.RandomState(7)
    g = sc["geometry"]
    g["position"][:] = rs.uniform(-1.0, 1.0, (len(g), 3)).astype(np.float32)
    g["radius_sq"][:] = (rs.uniform(5.0, 6.0, len(g)).astype(np.float32)) ** 2
    lights = np.arange(0, len(g), 64)  # the emissive spheres: small, on a shell around the cluster, so that shadow rays are traced too
    d = rs.randn(len(lights), 3); d /= np.linalg.norm(d, axis=1, keepdims=True)
    g["position"][lights] = (40.0 * d).astype(np.float32); g["radius_sq"][lights] = np.float32(4.0)
    sc["camera"] = dict(eye=(0, 2, 30), dir=(0, -0.05, -1), focal_length=50.0, exposure=1.0)
    w, h, mb = 96, 64, 4
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=b2r.FLAG_FORCE_BVH); r.Accumulate(2)
    _, max_stack = r.wide_nodes()
    assert max_stack > 13, max_stack  # deeper than the shared-memory stack minus its three slots of headroom
    o = oracle_for(sc, w, h, mb, 1); o.accumulate(2)
    frac = divergent_fraction(r.buckets_host(), o.buckets())
    gc, oc = r.counters(), o.counters()
    print(f"nested spheres: worst-case stack {max_stack}, divergent pixel fraction {frac:.3e}, rays {gc['extension_rays']}/{oc['extension_rays']}, shadow rays {gc['shadow_rays']}")
    assert r.buckets_host().tobytes() == o.buckets().tobytes() and gc["shadow_rays"] > 1000
    assert gc["extension_rays"] == oc["extension_rays"]
    r.close()


@pytest.mark.parametrize("w,h,tag", [(1920, 1088, "C3"), (3840, 2160, "C5")])
def test_bvh_equals_brute_on_gpu_at_full_size(w, h, tag):
    """Size-independent property at BASELINE's full sizes: on the GPU, BVH traversal and brute force over all 100k spheres give the same
    image for the same sample — the WHOLE C3 frame (1920x1088) and the whole C5 frame (3840x2160), one sample each (brute force over 1e5
    spheres is ~1e13 sphere tests per 4K sample: seconds on the GPU, hours on the CPU). The leaves' boxes are sized for the noise of the
    float sphere tests (leaf_half_extent), so the two agree bit for bit; the north_star divergent fraction is printed."""
    sc = scenes.random_scene(100000)
    ps = b2r.PreparedScene(sc, w, h)
    a = b2r.Renderer(ps, w, h, max_bounces=16, buckets=1, flags=b2r.FLAG_FORCE_BVH, samples_in_flight=1); a.Accumulate(1)
    b = b2r.Renderer(ps, w, h, max_bounces=16, buckets=1, flags=b2r.FLAG_FORCE_BRUTE, samples_in_flight=1); b.Accumulate(1)
    ga, gb = a.buckets_host(), b.buckets_host()
    frac = divergent_fraction(ga, gb); same = ga.tobytes() == gb.tobytes()
    ca, cb = a.counters(), b.counters()
    print(f"{tag} full frame {w}x{h}, 100k spheres, GPU BVH vs GPU brute force: divergent pixel fraction {frac:.3e}, bit-identical {same}; rays {ca['extension_rays']} vs {cb['extension_rays']}")
    assert same
    assert ca["extension_rays"] == cb["extension_rays"]
    a.close(); b.close()


def test_c3_full_size_oracle_spot_tiles():
    """BASELINE configs[2] at full size (100k spheres, 1920x1088 internal, MIS): 512 random 16x16 tiles (6 % of the frame) of two samples
    are re-rendered by the oracle (tiles are independent, Renderer.hpp:84) in stream-BVH mode and compared."""
    sc = scenes.random_scene(100000)
    w, h = 1920, 1088
    r = b2r.Renderer(sc, w, h, max_bounces=16, buckets=8, samples_in_flight=2); r.Accumulate(2)
    o = oracle_py.Oracle(w, h, max_bounces=16, K=8, flags=oracle_py.ORC_BVH, fast=True); o.set_scene(sc)   # same arithmetic contract (-ffp-contract=off), -O3
    tiles = np.random.RandomState(0).choice((w // 16) * (h // 16), 512, replace=False).astype(np.uint32)
    o.accumulate_tiles(tiles, 2, threads=os.cpu_count() or 1)
    g, ref = r.buckets_host(), o.buckets()
    idx = (tiles[:, None] * 256 + np.arange(256)[None, :]).ravel()
    frac = divergent_fraction(g[:, :, idx], ref[:, :, idx])
    print(f"C3 full-size spot tiles: divergent pixel fraction {frac:.3e} over {len(idx)} pixels, bit-identical {g[:, :, idx].tobytes() == ref[:, :, idx].tobytes()}")
    assert frac < 2e-4
    r.close(); o.close()


# ------------------------------------------------------------------------------------------------ interface behaviour
def test_white_furnace_known_answer():
    sc = scenes.white_furnace()
    r = b2r.Renderer(sc, 64, 48, max_bounces=16, buckets=1); r.Accumulate(3)
    assert np.all(r.buckets_host() == 3.0)
    r.close()


def test_sample_ranges_are_additive_and_resumable():
    """RNG is a pure function of (sample index, pixel, bounce) (Q2-Q3): rendering samples 1..10 at once, in pieces, with a
    different batch width, or after a bucket checkpoint restore gives identical bucket sums; graph and non-graph launches agree."""
    sc = scenes.default_scene(); w, h = 256, 144
    a = b2r.Renderer(sc, w, h, max_bounces=8, buckets=5); a.Accumulate(10); A = a.buckets_host()
    b = b2r.Renderer(sc, w, h, max_bounces=8, buckets=5, samples_in_flight=3, flags=b2r.FLAG_NO_GRAPH)
    b.Accumulate(4); ck = b.buckets_host(); b.ResetAccumulator(); b.write_buckets(ck); b.accumulations = 4; b.Accumulate(6)
    assert A.tobytes() == b.buckets_host().tobytes()
    kt = b.kernel_times(); assert kt["bounce_brute"][1] > 0 and kt["bounce_brute"][0] > 0.0
    a.ResetAccumulator(); assert a.accumulations == 0 and not a.buckets_host().any()
    a.Resize(128, 80); a.Accumulate(5); assert a.Render() and a.framebuffer.shape == (80, 128, 4)
    o = oracle_for(sc, 128, 80, 8, 5); o.accumulate(5)
    assert a.buckets_host().tobytes() == o.buckets().tobytes()
    a.close(); b.close()


def test_bucket_ownership_partitions_the_frame():
    """Multi-GPU split (SURVEY §8e): contexts owning buckets {b : b % G == g} together reproduce the single-context buckets."""
    sc = scenes.default_scene(); w, h, K = 192, 112, 8
    full = b2r.Renderer(sc, w, h, max_bounces=8, buckets=K); full.Accumulate(16); F = full.buckets_host()
    parts = np.zeros_like(F)
    for g in range(4):
        r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=K, bucket_first=g, bucket_stride=4); r.Accumulate(16)
        P = r.buckets_host()
        owned = [k for k in range(K) if k % 4 == g]
        assert not P[[k for k in range(K) if k not in owned]].any()
        parts += P; r.close()
    assert parts.tobytes() == F.tobytes()
    full.close()


def test_error_behaviour():
    sc = scenes.default_scene()
    with pytest.raises(b2r.B2RError) as e:
        b2r.Renderer(sc, 100, 64)
    assert e.value.code == b2r.ERR_ARG
    r = b2r.Renderer(None, 64, 64)
    with pytest.raises(b2r.B2RError) as e:
        r.Accumulate(1)
    assert e.value.code == b2r.ERR_STATE
    ps = b2r.PreparedScene(sc, 64, 64); bad = ps.nodes.copy(); bad["first_id"][0] = 0
    ps.nodes = bad
    with pytest.raises(b2r.B2RError) as e:
        r.SetScene(ps)
    assert e.value.code == b2r.ERR_BVH
    r.close()
    # B2R_FLAG_REFERENCE_EXACT is a create-time choice (it sizes the stream bookkeeping) and follows the reference's 64-material limit
    r = b2r.Renderer(sc, 64, 64)
    with pytest.raises(b2r.B2RError) as e:
        r.set_flags(b2r.FLAG_REFERENCE_EXACT)
    assert e.value.code == b2r.ERR_STATE
    r.close()
    many = scenes.random_scene(80, light_every=7)
    many["material"] = np.repeat(many["material"], 10, axis=0)[:70].copy()  # 70 materials > RendererPolicy::max_materialID
    r = b2r.Renderer(many, 64, 64, flags=b2r.FLAG_REFERENCE_EXACT | b2r.FLAG_FORCE_BRUTE)
    with pytest.raises(b2r.B2RError) as e:
        r.Accumulate(1)
    assert e.value.code == b2r.ERR_STATE
    r.close()


def test_cpp_mirror_frame_loop(tmp_path):
    """examples/frame_loop.cpp = the reference's per-frame driver (Application.cpp:361-406) on the C++ mirror
    (host/Renderer.hpp etc.): builds with g++, links libb2r.so, and must land on the same frame as the Python path."""
    import re
    import subprocess
    from conftest import ROOT, PKG
    exe = str(tmp_path / "frame_loop")
    subprocess.check_call(["g++", "-std=c++20", "-O2", os.path.join(ROOT, "examples", "frame_loop.cpp"), "-I", os.path.join(PKG, "host"),
                           "-L", PKG, "-lb2r", f"-Wl,-rpath,{PKG}", "-o", exe])
    out = subprocess.check_output([exe, "250", "130", "5"], text=True)   # padded to 256x144 like Application.cpp:367-372
    fp = re.search(r"focus pick: prim (-?\d+) mat (-?\d+) depth ([0-9.]+) \(renderer path: prim (-?\d+) depth ([0-9.]+)\)", out)
    assert fp and int(fp.group(1)) == int(fp.group(4)) >= 0 and fp.group(3) == fp.group(5)  # BVH::Traverse<8> == Renderer::Traverse
    m = re.search(r"\[(\d+) X (\d+)\].*mean tonemapped value ([0-9.]+) after (\d+) accumulations", out)
    assert m and (int(m.group(1)), int(m.group(2)), int(m.group(4))) == (256, 144, 5)
    r = b2r.Renderer(scenes.default_scene(), 256, 144, max_bounces=16, buckets=5); r.Accumulate(5); assert r.Render()
    assert abs(float(m.group(3)) - float(r.framebuffer[..., :3].mean(dtype=np.float64))) < 1e-5
    # the geometry drag at the end of the example (SceneMoved -> b2r_refit_scene) lands on the frame of a fresh upload of the moved scene
    e = re.search(r"after a geometry drag: tree quality ratio ([0-9.]+), mean tonemapped value ([0-9.]+) after (\d+) accumulations", out)
    assert e and int(e.group(3)) == 5 and float(e.group(1)) > 0.5
    sc = scenes.default_scene(); sc["geometry"]["position"][1, 0] += np.float32(0.25); sc["geometry"]["position"][1, 1] += np.float32(0.125)
    r.SetScene(sc); r.ResetAccumulator(); r.Accumulate(5); assert r.Render()
    assert abs(float(e.group(2)) - float(r.framebuffer[..., :3].mean(dtype=np.float64))) < 1e-5
    # ... and the edit that adds a sphere goes through SceneMoved()'s fallback to a full upload
    a = re.search(r"after adding a sphere: (\d+) spheres, tree quality ratio ([0-9.]+), mean tonemapped value ([0-9.]+) after (\d+) accumulations", out)
    assert a and int(a.group(1)) == 10 and float(a.group(2)) == 1.0 and int(a.group(4)) == 5
    mat = np.zeros(1, scenes.MATERIAL_DTYPE); mat["albedo"] = (0.2, 0.6, 0.3)
    sph = np.zeros(1, scenes.SPHERE_DTYPE); sph["position"] = (0.125, 0.0625, 0.375); sph["radius_sq"] = np.float32(0.0625) * np.float32(0.0625); sph["material_ID"] = 9
    sc["material"] = np.concatenate([sc["material"], mat]); sc["geometry"] = np.concatenate([sc["geometry"], sph])
    r.SetScene(sc); r.ResetAccumulator(); r.Accumulate(5); assert r.Render()
    assert abs(float(a.group(3)) - float(r.framebuffer[..., :3].mean(dtype=np.float64))) < 1e-5
    r.close()


@pytest.mark.parametrize("n,K,mb,flags", [(1, 1, 1, 0), (2, 3, 2, 0), (33, 5, 4, 0), (33, 64, 3, b2r.FLAG_FORCE_BRUTE), (1500, 7, 5, b2r.FLAG_FORCE_BRUTE), (9, 8, 40, 0)])
def test_edge_configurations(n, K, mb, flags):
    """Smallest scenes (single sphere = single-leaf tree), the 32/33-sphere brute/BVH switch, multi-tile brute force (1500 > 1024
    spheres per shared-memory tile), extreme bucket counts (1, 64) and bounce limits (1, 40), ragged batches (n_samples not a
    multiple of the batch width): bucket sums bit-exact vs the oracle."""
    sc = scenes.default_scene() if n == 9 else scenes.random_scene(n, light_every=max(1, n // 3))
    w, h = 96, 64
    samples = K + 3 if K < 20 else K
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=flags, samples_in_flight=5); r.Accumulate(samples)
    o = oracle_for(sc, w, h, mb, K); o.accumulate(samples)
    g, ref = r.buckets_host(), o.buckets()
    frac = divergent_fraction(g, ref)
    assert frac == 0.0 and g.tobytes() == ref.tobytes(), (n, K, mb, frac)
    r.accumulations = (samples // K) * K
    if r.accumulations:
        o.set_accumulations(r.accumulations)
        assert r.Render() and r.framebuffer.tobytes() == o.render()[1].tobytes()
    r.close()


# ------------------------------------------------------------------------------------------------ GGX closure (B2R_FLAG_GGX)
@pytest.mark.parametrize("name,flags,w,h,mb,K,n", [("default", 0, 320, 192, 16, 5, 10), ("default", b2r.FLAG_FORCE_BVH, 160, 96, 8, 5, 7), ("brdf_test", 0, 160, 96, 8, 5, 5),
                                                  ("ggx_random", b2r.FLAG_FORCE_BRUTE, 128, 80, 8, 4, 8), ("ggx_random", 0, 128, 80, 8, 4, 8)])
def test_ggx_closure_matches_oracle(name, flags, w, h, mb, K, n):
    """The reference's `#define BRDF 1` build (Closure<GGX>, DataStreams.hpp:184-219) on the GPU: both pipelines, every kernel that shades
    (k_bounce_brute, k_brute_finish, k_shade), against the oracle's ORC_GGX mode, which tests/test_oracle_ref_renderer.py pins bit for bit to
    the reference's own Renderer<> built that way. Brute-force pipeline: bit-exact bucket sums and frame; BVH pipeline: bit-exact whenever its
    hit decisions equal brute force (asserted: 0 divergent pixels on these scenes)."""
    sc = {"default": scenes.default_scene, "brdf_test": scenes.brdf_test_scene, "ggx_random": lambda: scenes.ggx_random_scene(1500, light_every=40)}[name]()
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=flags | b2r.FLAG_GGX, samples_in_flight=3); r.Accumulate(n)
    o = oracle_for(sc, w, h, mb, K, flags=oracle_py.ORC_GGX); o.accumulate(n)
    g, ref = r.buckets_host(), o.buckets()
    frac = divergent_fraction(g, ref)
    print(f"GGX {name} flags={flags}: divergent pixel fraction {frac:.3e}, bit-exact {g.tobytes() == ref.tobytes()}")
    assert np.isfinite(g).all() and frac == 0.0 and g.tobytes() == ref.tobytes()
    lam = oracle_for(sc, w, h, mb, K); lam.accumulate(n)
    assert lam.buckets().tobytes() != g.tobytes()  # not the Lambertian image
    if n % K == 0:
        assert r.Render() and r.framebuffer.tobytes() == o.render()[1].tobytes()
    r.close()


def test_ggx_closure_full_batches_and_flag_rules():
    """Full-width batches (twin lanes, k_brute_finish hand-over) give the same bits as narrow ones; GGX cannot be combined with the
    reference-exact stream bookkeeping; the closure can be switched per frame with b2r_set_flags."""
    sc = scenes.default_scene(); w, h, mb, K = 640, 368, 16, 8
    a = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=b2r.FLAG_GGX); a.Accumulate(16)
    b = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=b2r.FLAG_GGX | b2r.FLAG_NO_GRAPH, samples_in_flight=1); b.Accumulate(16)
    assert a.buckets_host().tobytes() == b.buckets_host().tobytes()
    b.close()
    with pytest.raises(b2r.B2RError) as e:
        b2r.Renderer(sc, 64, 64, flags=b2r.FLAG_GGX | b2r.FLAG_REFERENCE_EXACT)
    assert e.value.code == b2r.ERR_ARG
    a.set_flags(0); a.ResetAccumulator(); a.Accumulate(8)
    o = oracle_for(sc, w, h, mb, K); o.accumulate(8)
    assert a.buckets_host().tobytes() == o.buckets().tobytes()
    a.close()


@pytest.mark.skipif(not oracle_py.have_reference_renderer(ggx=True), reason="oracle/_ref/librefrenderer_ggx.so not present")
def test_ggx_closure_vs_the_references_own_brdf1_build_live():
    """GPU against the reference itself built with `#define BRDF 1`, run here on the host cores: per-sample radiance within 1e-4 relative
    except the (reported) fraction of pixels whose ray sat in a scalar-tail slot of the reference's SIMD loop (DESIGN.md section 2)."""
    sc = scenes.default_scene(); w, h, mb = 640, 368, 8
    ref = oracle_py.ReferenceRenderer(sc, w, h, mb, ggx=True); ref.accumulate(1); ref_first = ref.buckets()[1].copy(); ref.close()
    g = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=b2r.FLAG_GGX); g.Accumulate(1)
    mine = g.buckets_host()[1]
    frac = divergent_fraction(mine, ref_first)
    exact = float((mine.view(np.uint32) == ref_first.view(np.uint32)).all(axis=0).mean())
    print(f"GGX: GPU vs the reference's BRDF 1 build: divergent pixel fraction {frac:.3e}, bit-identical pixels {exact:.4f}")
    assert frac < 2e-3 and exact > 0.99
    g.close()


def test_no_mis_variant_matches_oracle_definition():
    sc = scenes.default_scene()
    r = b2r.Renderer(sc, 160, 96, max_bounces=8, buckets=1, flags=b2r.FLAG_NO_MIS); r.Accumulate(2)
    o = oracle_for(sc, 160, 96, 8, 1, flags=oracle_py.ORC_NO_MIS); o.accumulate(2)
    assert r.buckets_host().tobytes() == o.buckets().tobytes() and r.counters()["shadow_rays"] == 0
    r.close()


def test_c2_full_size_bit_exact():
    """BASELINE configs[1] at FULL size: default scene, 1920x1080 rendered as 1920x1088 (SURVEY F6), 64 spp, 8 buckets,
    max_bounces 16 — bucket sums and the tonemapped frame bit-exact against the oracle (timing build, proven bit-identical to the
    parity build by tests/test_oracle_kat.py); cropped 1080-row RMSE reported."""
    sc = scenes.default_scene(); w, h, K = 1920, 1088, 8
    r = b2r.Renderer(sc, w, h, max_bounces=16, buckets=K); r.Accumulate(64); assert r.Render()
    o = oracle_py.Oracle(w, h, max_bounces=16, K=K, fast=True); o.set_scene(sc); o.accumulate(64)
    g, ref = r.buckets_host(), o.buckets()
    frac = divergent_fraction(g, ref)
    rc, img = o.render()
    rmse = float(np.sqrt(np.mean((r.framebuffer[:1080] - img[:1080]) ** 2)))
    print(f"C2 full size: divergent pixel fraction {frac:.3e}, bit-exact buckets {g.tobytes() == ref.tobytes()}, frame RMSE {rmse:.3e}")
    assert g.tobytes() == ref.tobytes() and r.framebuffer.tobytes() == img.tobytes() and rmse < 1e-3
    gc, oc = r.counters(), o.counters()
    assert gc["extension_rays"] == oc["extension_rays"] and gc["terminated"] == oc["terminated"] and gc["dropped"] == oc["dropped"]
    r.close()


@pytest.mark.parametrize("flags", [b2r.FLAG_FORCE_BRUTE, b2r.FLAG_FORCE_BVH])
def test_sky_hdri_scene(flags):
    """SURVEY §8f row 1: the miss shader with an equirect HDRI (Renderer.hpp:411-420, Primitives.hpp:35-46, fast_atan2/fast_asin),
    on Scenes::BVH_test as the reference lights it (ambient 1): both pipelines bit-exact vs the oracle, Q14 included."""
    sc = scenes.bvh_test_scene(255)
    r = b2r.Renderer(sc, 256, 144, max_bounces=8, buckets=5, flags=flags); r.Accumulate(5); assert r.Render()
    o = oracle_for(sc, 256, 144, 8, 5); o.accumulate(5)
    g, ref = r.buckets_host(), o.buckets()
    assert divergent_fraction(g, ref) == 0.0 and g.tobytes() == ref.tobytes()
    assert r.framebuffer.tobytes() == o.render()[1].tobytes()
    r.close()


@pytest.mark.parametrize("flags", [0, b2r.FLAG_FORCE_BVH, b2r.FLAG_REFERENCE_EXACT])
def test_brdf_test_scene(flags):
    """Scenes::BRDF_test as shipped (Application.cpp:123-217; albedo-0 spheres under the Lambertian closure: zero throughput, roulette
    q = 1, Q13), ambient HDRI sky: bit-exact vs the oracle in canonical mode; in reference-exact mode vs the oracle's slot-exact mode,
    which tests/test_oracle_ref_renderer.py pins to the reference's own renderer on this scene."""
    sc = scenes.brdf_test_scene()
    exact = bool(flags & b2r.FLAG_REFERENCE_EXACT)
    r = b2r.Renderer(sc, 192, 112, max_bounces=8, buckets=5, flags=flags); r.Accumulate(10); assert r.Render()
    o = oracle_for(sc, 192, 112, 8, 5, flags=oracle_py.ORC_SLOT_EXACT if exact else 0); o.accumulate(10)
    g, ref = r.buckets_host(), o.buckets()
    assert g.tobytes() == ref.tobytes() and r.framebuffer.tobytes() == o.render()[1].tobytes()
    c = r.counters(); assert c["shaded_hits"] > 0 and c["shadow_rays"] > 0 and float(g.max()) > 0.0
    r.close()


def test_sky_loaded_from_a_radiance_file(tmp_path):
    """The sky as the reference gets it (Application.cpp:225-231): an .hdr file decoded by b2r_read_hdr (stb_image's Radiance decoder
    restated) and handed to b2r_upload_scene. RGBE keeps 8 mantissa bits, so the oracle is given the same decoded array: bit-exact."""
    tex = scenes.synthetic_hdri(96, 48, seed=3)
    b2r.write_hdr(tmp_path / "env.hdr", tex[::-1])      # the writer flips rows (Image.cpp:72): store it so that the file holds `tex` top-down
    env = b2r.read_hdr(tmp_path / "env.hdr")
    assert env.shape == tex.shape and np.all(np.abs(env[..., :3] - tex[..., :3]) <= tex[..., :3].max(axis=2, keepdims=True) / 128)
    sc = scenes.bvh_test_scene(255, hdri=env)
    r = b2r.Renderer(sc, 128, 80, max_bounces=8, buckets=5); r.Accumulate(5); assert r.Render()
    o = oracle_for(sc, 128, 80, 8, 5); o.accumulate(5)
    assert r.buckets_host().tobytes() == o.buckets().tobytes() and r.framebuffer.tobytes() == o.render()[1].tobytes()
    assert float(r.buckets_host().max()) > 0.0
    r.close()


def test_c4_size_oracle_spot_tiles():
    """BASELINE configs[3] size (1M spheres, 3840x2160, max_bounces 16): one sample, 24 random tiles re-rendered by the oracle in
    stream-BVH mode. Also exercises the 22-bit node index / 13-bit distance split of the traversal stack entries."""
    sc = scenes.random_scene(1000000)
    w, h = 3840, 2160
    r = b2r.Renderer(sc, w, h, max_bounces=16, buckets=8, samples_in_flight=1); r.Accumulate(1)
    wide, max_stack = r.wide_nodes()
    assert max_stack + 3 <= 64 and len(wide) < (1 << 22)
    o = oracle_for(sc, w, h, 16, 8, flags=oracle_py.ORC_BVH)
    tiles = np.random.RandomState(4).choice((w // 16) * (h // 16), 24, replace=False).astype(np.uint32)
    o.accumulate_tiles(tiles, 1)
    g, ref = r.buckets_host(), o.buckets()
    idx = (tiles[:, None] * 256 + np.arange(256)[None, :]).ravel()
    frac = divergent_fraction(g[:, :, idx], ref[:, :, idx])
    print(f"C4-size spot tiles: divergent pixel fraction {frac:.3e} over {len(idx)} pixels; {len(wide)} wide nodes, stack bound {max_stack}")
    assert frac < 5e-3
    r.close()


def test_randomised_configurations_bit_exact():
    """Fuzz: random scenes (sizes on both sides of the brute/BVH switch), cameras, image sizes, bucket counts, bounce limits,
    batch widths and starting sample indices — bucket sums must equal the oracle's bit for bit every time."""
    rs = np.random.RandomState(20261018)
    for trial in range(12):
        n = int(rs.choice([3, 9, 31, 32, 33, 60, 200, 700]))
        sc = scenes.random_scene(n, light_every=int(rs.randint(1, max(2, n // 2))), seed=int(rs.randint(1, 2 ** 31)))
        eye = rs.uniform([-150, 10, 150], [150, 90, 320]); look = np.array([0.0, 40.0, 0.0]) - eye
        sc["camera"] = dict(eye=tuple(eye), dir=tuple(look), focal_length=float(rs.uniform(20, 80)), exposure=float(rs.uniform(0.5, 2.0)))
        if rs.rand() < 0.4:
            sc["ambient"] = tuple(rs.uniform(0.0, 1.0, 3)); sc["hdri"] = scenes.synthetic_hdri(int(rs.randint(1, 40)), int(rs.randint(1, 20)), seed=trial)
        w, h = 16 * int(rs.randint(1, 9)), 16 * int(rs.randint(1, 7))
        K, mb, sif = int(rs.randint(1, 10)), int(rs.randint(1, 20)), int(rs.randint(1, 9))
        start, samples = int(rs.randint(0, 5000)), int(rs.randint(1, 12))
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, samples_in_flight=sif); r.accumulations = start; r.Accumulate(samples)
        o = oracle_for(sc, w, h, mb, K); o.set_accumulations(start); o.accumulate(samples)
        g, ref = r.buckets_host(), o.buckets()
        assert g.tobytes() == ref.tobytes(), dict(trial=trial, n=n, w=w, h=h, K=K, mb=mb, sif=sif, start=start, samples=samples, frac=divergent_fraction(g, ref))
        r.close()


def test_c3_converged_image_at_reduced_size():
    """BASELINE configs[2] semantics (100k-sphere scene, 16 spp, K = 8, NEE + MIS, max_bounces 16) at 480x272: the resolved,
    tonemapped frame against the CPU oracle (stream-BVH restatement of BVH.hpp:320-358) — RMSE < 1e-3, divergent fraction reported."""
    sc = scenes.random_scene(100000); w, h, K = 480, 272, 8
    r = b2r.Renderer(sc, w, h, max_bounces=16, buckets=K); r.Accumulate(16); assert r.Render()
    o = oracle_py.Oracle(w, h, max_bounces=16, K=K, flags=oracle_py.ORC_BVH, fast=True); o.set_scene(sc); o.accumulate(16)
    rc, img = o.render(); assert rc == 0
    frac = divergent_fraction(r.buckets_host(), o.buckets())
    rmse = float(np.sqrt(np.mean((r.framebuffer - img) ** 2)))
    lin = np.zeros_like(r.framebuffer); assert r.Render(tonemap=False, out=lin)
    rmse_lin = float(np.sqrt(np.mean((lin - o.render(tonemap=False)[1]) ** 2)))
    print(f"C3 scene 480x272 16 spp: divergent pixel fraction {frac:.3e}, tonemapped RMSE {rmse:.3e}, linear RMSE {rmse_lin:.3e}")
    assert rmse < 1e-3 and frac < 5e-3
    r.close()


# ------------------------------------------------------------------------------------------------ against the reference itself
def test_gpu_vs_reference_renderer_fixture():
    """north_star's correctness check, literally: the GPU against the reference's own CPU Renderer::Accumulate / Render on the same scene,
    camera, seeds and bounce count. The reference's outputs (oracle/_ref/librefrenderer.so, built from /root/reference by
    oracle/ref_renderer_build.sh) are committed as tests/golden/reference_default_160x96_mb16.npz by tests/gen_golden.py."""
    ref = np.load(os.path.join(G, "reference_default_160x96_mb16.npz"))
    sc = scenes.default_scene(); w, h, mb = 160, 96, 16
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5)
    r.Accumulate(1)
    frac = divergent_fraction(r.buckets_host()[1], ref["first_sample"])
    r.Accumulate(199); assert r.Render()
    rmse = float(np.sqrt(np.mean((r.framebuffer[..., :3] - ref["frame_200spp"][..., :3]) ** 2)))
    print(f"GPU vs the reference's Renderer (default scene 160x96, max_bounces 16): divergent per-sample pixel fraction {frac:.3e}, 200-spp tonemapped RMSE {rmse:.3e}")
    assert frac < 2e-3 and rmse < 1e-3
    r.close()


@pytest.mark.skipif(not oracle_py.have_reference_renderer(), reason="oracle/_ref/librefrenderer.so not present")
def test_c1_full_size_gpu_vs_reference_renderer_live():
    """BASELINE config C1 (default scene, 1280x720, 1 spp, max_bounces 8) on the GPU and through the reference's own Renderer::Accumulate
    run here on the host cores; then 4 more samples and Renderer::Render (median of 5 + ACES) on both."""
    sc = scenes.default_scene(); w, h, mb = 1280, 720, 8
    ref = oracle_py.ReferenceRenderer(sc, w, h, mb); ref.accumulate(1); ref_first = ref.buckets()[1].copy()
    g = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5); g.Accumulate(1)
    frac = divergent_fraction(g.buckets_host()[1], ref_first)
    exact = float((g.buckets_host()[1].view(np.uint32) == ref_first.view(np.uint32)).all(axis=0).mean())
    ref.accumulate(4); acted, ref_frame = ref.render(); ref.close()
    g.Accumulate(4); assert g.Render() and acted
    rmse = float(np.sqrt(np.mean((g.framebuffer[..., :3] - ref_frame[..., :3]) ** 2)))
    print(f"C1 GPU vs the reference itself: divergent pixel fraction {frac:.3e} (bit-identical pixels {exact:.4f}), 5-spp frame RMSE {rmse:.3e}")
    assert frac < 2e-3 and rmse < 5e-3  # 5 samples are far from converged: a divergent path moves its pixel visibly; the converged bound is tested above
    g.close()


def test_reference_binding_dropin_on_the_references_own_scene():
    """include/b2r_reference_binding.hpp — the binding a maintainer would add (INTEGRATION.md §1) — compiled against the reference's own
    headers: tests/refbinding builds ONE reference `Scene`, renders it with the reference's `Renderer<>` on the host and with
    `b2r::ReferenceRenderer` on the GPU, through the same call sequence as the app's frame loop, and compares the framebuffers."""
    import subprocess
    exe = os.path.join(os.path.dirname(__file__), "refbinding", "refbinding")
    if not os.path.exists(exe):
        pytest.skip("tests/refbinding/refbinding not present (built only where /root/reference exists)")
    p = subprocess.run([exe, "200"], capture_output=True, text=True, timeout=600)
    print(p.stdout.strip()); print(p.stderr.strip()[-2000:])
    assert p.returncode == 0 and "REFBINDING OK" in p.stdout
    # with B2R_FLAG_REFERENCE_EXACT the drop-in's framebuffer is the reference's, bit for bit, at every compared frame
    p = subprocess.run([exe, "100", "exact"], capture_output=True, text=True, timeout=600)
    print(p.stdout.strip()); print(p.stderr.strip()[-2000:])
    assert p.returncode == 0 and "REFBINDING OK" in p.stdout and "bit-identical: yes" in p.stdout


# ------------------------------------------------------------------------------------------------ bit-exact against the reference itself
@pytest.mark.parametrize("name,w,h,mb,n,first,sif", [("default", 160, 96, 16, 10, 0, 0), ("default", 64, 48, 8, 5, 0, 1), ("default", 96, 64, 16, 7, 60, 3),
                                                     ("random33", 80, 48, 8, 5, 0, 0), ("random300_brute", 64, 48, 4, 5, 0, 0), ("sky", 64, 48, 8, 5, 0, 2)])
def test_reference_exact_mode_equals_slot_exact_oracle(name, w, h, mb, n, first, sif):
    """B2R_FLAG_REFERENCE_EXACT: the GPU reproduces the reference's slot-dependent choice of sphere formula (scalar tail for the last
    `active % 8` rays of each tile stream, stream order = stable counting sort by material). Bit-exact against the oracle's slot-exact
    mode, which is itself bit-exact against the reference's own Renderer (tests/test_oracle_ref_renderer.py)."""
    sc = {"default": scenes.default_scene, "random33": lambda: scenes.random_scene(33, light_every=3), "random300_brute": lambda: scenes.random_scene(300, light_every=20),
          "sky": lambda: scenes.bvh_test_scene(40, hdri=scenes.synthetic_hdri())}[name]()
    flags = b2r.FLAG_REFERENCE_EXACT | b2r.FLAG_FORCE_BRUTE
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=flags, samples_in_flight=sif)
    o = oracle_for(sc, w, h, mb, 5, flags=oracle_py.ORC_SLOT_EXACT)
    if first:
        r.accumulations = first; o.set_accumulations(first)
    r.Accumulate(n); o.accumulate(n)
    gb, ob = r.buckets_host(), o.buckets()
    assert gb.tobytes() == ob.tobytes(), f"{name}: {float((gb.view(np.uint32) != ob.view(np.uint32)).any(axis=(0, 1)).mean()):.3e} of pixels differ"
    if (first + n) % 5 == 0:
        rc, of = o.render(); assert r.Render() and rc == 0
        assert r.framebuffer.tobytes() == of.tobytes()
    r.close(); o.close()


@pytest.mark.skipif(not oracle_py.have_reference_renderer(), reason="oracle/_ref/librefrenderer.so not present")
def test_c1_full_size_reference_exact_mode_bit_identical_to_the_reference():
    """BASELINE config C1 at full size, GPU in B2R_FLAG_REFERENCE_EXACT mode against the reference's own Renderer::Accumulate / Render
    run live on the host cores: all five bucket planes and the tonemapped frame must be identical bit for bit."""
    sc = scenes.default_scene(); w, h, mb = 1280, 720, 8
    ref = oracle_py.ReferenceRenderer(sc, w, h, mb); ref.accumulate(5); rb = ref.buckets(); acted, rframe = ref.render(); ref.close()
    g = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=b2r.FLAG_REFERENCE_EXACT); g.Accumulate(5)
    gb = g.buckets_host()
    same = float((gb.view(np.uint32) == rb.view(np.uint32)).all(axis=(0, 1)).mean())
    print(f"C1, reference-exact mode vs the reference itself: bit-identical pixels {same:.6f}")
    assert gb.tobytes() == rb.tobytes()
    assert g.Render() and acted and g.framebuffer.tobytes() == rframe.tobytes()
    g.close()


@pytest.mark.skipif(not oracle_py.have_reference_renderer(), reason="oracle/_ref/librefrenderer.so not present")
def test_c2_size_reference_exact_mode_bit_identical_to_the_reference():
    """BASELINE config C2's frame (1920x1080 -> 1920x1088, max_bounces 16) with the reference's own estimator (K = 5, 65 samples: the
    reference-exact variant of SURVEY §8d) — 136M paths through the reference's Renderer on the host cores and through the GPU in
    B2R_FLAG_REFERENCE_EXACT mode: bucket sums and the tonemapped frame identical bit for bit."""
    sc = scenes.default_scene(); w, h, mb, n = 1920, 1088, 16, 65
    ref = oracle_py.ReferenceRenderer(sc, w, h, mb); ref.accumulate(n); rb = ref.buckets(); acted, rframe = ref.render(); ref.close()
    g = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=b2r.FLAG_REFERENCE_EXACT); g.Accumulate(n)
    gb = g.buckets_host()
    same = float((gb.view(np.uint32) == rb.view(np.uint32)).all(axis=(0, 1)).mean())
    print(f"C2 frame, K=5, 65 spp, reference-exact mode vs the reference itself: bit-identical pixels {same:.6f}")
    assert gb.tobytes() == rb.tobytes()
    assert g.Render() and acted and g.framebuffer.tobytes() == rframe.tobytes()
    g.close()


@pytest.mark.parametrize("n,w,h,mb,spp", [(600, 96, 64, 8, 5), (5000, 80, 48, 16, 5)])
def test_reference_exact_mode_bvh_pipeline_equals_slot_exact_oracle(n, w, h, mb, spp):
    """B2R_FLAG_REFERENCE_EXACT through the flattened-BVH kernels: tail rays take the scalar formula in the leaf tests, k_shade leaves
    (material, slot) behind, k_stream_rank orders the next bounce — against the oracle's slot-exact BRUTE-FORCE mode (the semantics the
    reference ships). Bit-exact: the BVH's hit decisions equal brute force for the scalar-tail formula too (tests/test_traversal_exact.py)."""
    sc = scenes.random_scene(n, light_every=40)
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=b2r.FLAG_REFERENCE_EXACT | b2r.FLAG_FORCE_BVH); r.Accumulate(spp)
    o = oracle_for(sc, w, h, mb, 5, flags=oracle_py.ORC_SLOT_EXACT); o.accumulate(spp)
    gb, ob = r.buckets_host(), o.buckets()
    same = float((gb.view(np.uint32) == ob.view(np.uint32)).all(axis=(0, 1)).mean())
    print(f"BVH pipeline, reference-exact mode, n={n}: bit-identical pixels {same:.6f}, divergent fraction {divergent_fraction(gb, ob):.3e}")
    assert gb.tobytes() == ob.tobytes()
    r.close(); o.close()


@pytest.mark.skipif(not oracle_py.have_reference_renderer(), reason="oracle/_ref/librefrenderer.so not present")
def test_bvh_pipeline_reference_exact_mode_vs_the_reference_itself():
    """2000 random spheres (the reference brute-forces them on the host cores), GPU through the BVH kernels in reference-exact mode."""
    sc = scenes.random_scene(2000, light_every=100); w, h, mb = 96, 64, 16
    ref = oracle_py.ReferenceRenderer(sc, w, h, mb); ref.accumulate(5); rb = ref.buckets(); acted, rframe = ref.render(); ref.close()
    g = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=b2r.FLAG_REFERENCE_EXACT | b2r.FLAG_FORCE_BVH); g.Accumulate(5)
    gb = g.buckets_host()
    same = float((gb.view(np.uint32) == rb.view(np.uint32)).all(axis=(0, 1)).mean())
    print(f"2000 spheres, BVH kernels in reference-exact mode vs the reference itself: bit-identical pixels {same:.6f}")
    assert same > 0.998 and divergent_fraction(gb, rb) < 2e-3
    if same == 1.0:
        assert g.Render() and acted and g.framebuffer.tobytes() == rframe.tobytes()
    g.close()


@pytest.mark.skipif(not oracle_py.have_reference_renderer(), reason="oracle/_ref/librefrenderer.so not present")
def test_c3_scene_reference_exact_mode_vs_the_reference_itself():
    """BASELINE config C3's scene (100k random spheres, 100 lights, max_bounces 16, its camera) on a 64x48 frame: the reference
    brute-forces 100k spheres per ray on the host cores (a few seconds); the GPU walks its BVH in reference-exact mode."""
    sc = scenes.random_scene(100000); w, h, mb = 64, 48, 16
    ref = oracle_py.ReferenceRenderer(sc, w, h, mb); ref.accumulate(5); rb = ref.buckets(); acted, rframe = ref.render(); ref.close()
    g = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=5, flags=b2r.FLAG_REFERENCE_EXACT); g.Accumulate(5)
    gb = g.buckets_host()
    same = float((gb.view(np.uint32) == rb.view(np.uint32)).all(axis=(0, 1)).mean())
    print(f"C3 scene (100k spheres) 64x48, BVH kernels in reference-exact mode vs the reference itself: bit-identical pixels {same:.6f}, divergent fraction {divergent_fraction(gb, rb):.3e}")
    assert same > 0.998 and divergent_fraction(gb, rb) < 2e-3
    if same == 1.0:
        assert g.Render() and acted and g.framebuffer.tobytes() == rframe.tobytes()
    g.close()


def test_async_resolve_delivers_the_same_frames():
    """b2r_resolve_async / b2r_frame_wait: three frames rendered back to back, each copied out on the second stream while the next
    one is traced, equal the frames of the synchronous Render() bit for bit."""
    import torch
    sc = scenes.default_scene(); w, h, mb, K = 320, 192, 8, 5
    a = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K); b = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K)
    pinned = [torch.empty((h, w, 4), dtype=torch.float32, pin_memory=True).numpy() for _ in range(3)]
    sync_frames = []
    for i in range(3):
        a.Accumulate(K); assert a.Render(); sync_frames.append(a.framebuffer.copy())
        b.Accumulate(K); assert b.RenderAsync(pinned[i])
    b.WaitFrame()
    for i in (0, 1, 2):
        assert pinned[i].tobytes() == sync_frames[i].tobytes()
    b.Accumulate(1)
    assert not b.RenderAsync(pinned[1])  # accumulations % K != 0: no-op like Renderer::Render (Renderer.hpp:437)
    a.close(); b.close()


@pytest.mark.parametrize("n,flags", [(9, 0), (3000, 0), (3000, b2r.FLAG_GGX)])
def test_frames_enqueued_back_to_back_equal_frames_waited_for(n, flags):
    """b2r_resolve_device: frames enqueued without a host wait are traced on alternating halves of the queue memory ("sides", on the library's
    own streams) while the previous frame's last bounces, fold and resolve still run — reset, fold and resolve stay on the caller's stream in
    call order. Buckets after every frame (read back once the pipeline has drained) and the frames themselves equal those of a renderer that
    waits after every call, bit for bit; a scene edit and a camera move between two pipelined frames land between exactly those frames."""
    sc = scenes.default_scene() if n == 9 else scenes.ggx_random_scene(n, light_every=30)
    w, h, mb, K = 256, 160, 8, 4
    a = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=flags); b = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=flags)
    rs = np.random.RandomState(3)
    geo2 = _moved_geometry(sc["geometry"], rs, jitter=0.3)
    sc2 = scenes.Scene(sc); sc2["geometry"] = geo2
    cam2 = dict(sc["camera"]); cam2["eye"] = tuple(np.asarray(cam2["eye"], np.float64) + np.array([0.05, 0.02, -0.1]))
    want = []
    for i in range(6):
        if i == 3: a.SetScene(b2r.PreparedScene(sc2, w, h))
        if i == 4: a.SetCamera(b2r.PreparedScene(dict(sc2, camera=cam2), w, h).camera)
        a.ResetAccumulator(); a.Accumulate(3 * K); assert a.Render(); a.sync(); want.append((a.buckets_host().copy(), a.framebuffer.copy()))
    got = []
    for i in range(6):  # nothing in this loop waits for the device
        if i == 3: b.SetScene(b2r.PreparedScene(sc2, w, h))
        if i == 4: b.SetCamera(b2r.PreparedScene(dict(sc2, camera=cam2), w, h).camera)
        b.ResetAccumulator(); b.Accumulate(3 * K); assert b.RenderDevice()
        if i in (2, 5):  # drain and look: the frame on the device is frame i
            b.sync(); bk = b.buckets_host().copy(); assert b.Render(); got.append((i, bk, b.framebuffer.copy()))
    for i, bk, fb in got:
        assert bk.tobytes() == want[i][0].tobytes() and fb.tobytes() == want[i][1].tobytes(), i
    b.Accumulate(1); assert not b.RenderDevice()  # accumulations % K != 0: no-op like Renderer::Render (Renderer.hpp:437)
    a.close(); b.close()


def test_a_scene_upload_every_frame_does_not_wait_for_the_frame_in_flight():
    """The e2e pattern, stressed: a DIFFERENT scene is uploaded (or refitted) before every frame and nothing waits for the device. Scene writes
    go to the library's upload stream while the previous frame still traces from its side's own copy of the scene arrays; every frame must
    still see exactly the scene uploaded before it. Two of the writes outgrow every scene before them (the upload of sc_e: more spheres,
    materials and lights; the refit to mat_f: more materials and lights), so the library's tables and the sides' copies are replaced while
    the previous frame may still be tracing."""
    w, h, mb, K = 192, 128, 6, 2
    sc_a = scenes.random_scene(2500, light_every=40); rs = np.random.RandomState(11)
    sc_b = scenes.Scene(sc_a); sc_b["geometry"] = _moved_geometry(sc_a["geometry"], rs, jitter=0.4)
    sc_c = scenes.random_scene(1800, light_every=25, seed=0x1234567)           # another sphere count: other array sizes, other tree
    geo_d = _moved_geometry(sc_a["geometry"], rs, jitter=0.2)                  # reached by a refit of sc_a
    sc_e = scenes.random_scene(3200, light_every=20, seed=0x2468ace)           # 3200 spheres, 160 lights
    extra = sc_e["material"][:4].copy(); extra["albedo"] *= 0.5
    sc_e["material"] = np.concatenate([sc_e["material"], extra])               # 13 materials, the last four on every seventh non-emissive sphere
    geo_e = sc_e["geometry"].copy(); pick = (np.arange(len(geo_e)) % 7 == 3) & (geo_e["material_ID"] < 8)
    geo_e["material_ID"][pick] = 9 + geo_e["material_ID"][pick] % 4; sc_e["geometry"] = geo_e
    geo_f = _moved_geometry(geo_e, rs, jitter=0.2)                             # reached by a refit of sc_e with mat_f:
    mat_f = np.concatenate([sc_e["material"], extra[:3]]); mat_f["emission"][0] = 2.0   # 16 materials, material 0's spheres become lights too
    plan = ["a", "b", "a", "c", "a", "refit_d", "b", "c", "e", "refit_f", "a"]
    def drive(r, wait):
        out = []
        for step in plan:
            if step == "refit_d": r.RefitScene(geo_d, want_quality=False)
            elif step == "refit_f": r.RefitScene(geo_f, material=mat_f, want_quality=False)
            else: r.SetScene(b2r.PreparedScene({"a": sc_a, "b": sc_b, "c": sc_c, "e": sc_e}[step], w, h))
            r.ResetAccumulator(); r.Accumulate(2 * K)
            if wait: assert r.Render(); out.append(r.buckets_host().copy())
            else: assert r.RenderDevice()
        return out
    a = b2r.Renderer(sc_a, w, h, max_bounces=mb, buckets=K); want = drive(a, True)
    for upto in (len(plan), 5, 6, 9, 10):   # drain after the whole plan, and after prefixes that end on other sides / other kinds of write
        b = b2r.Renderer(sc_a, w, h, max_bounces=mb, buckets=K)
        full = plan[:]; del plan[upto:]
        drive(b, False); b.sync()
        assert b.buckets_host().tobytes() == want[upto - 1].tobytes(), upto
        plan[:] = full; b.close()
    a.close()


# ------------------------------------------------------------------------------------------------ scene edit: GPU refit
def _moved_geometry(geo, rs, jitter=0.5, far=0):
    """Every sphere moves by up to `jitter` radii and changes radius by up to 20 %; `far` of them jump anywhere in the scene."""
    out = geo.copy(); r = np.sqrt(out["radius_sq"])
    out["position"] += (rs.uniform(-1, 1, (len(out), 3)) * (jitter * r)[:, None]).astype(np.float32)
    out["radius_sq"] = ((r * rs.uniform(0.8, 1.2, len(out))) ** 2).astype(np.float32)
    if far:
        idx = rs.choice(len(out), far, replace=False)
        lo, hi = geo["position"].min(0), geo["position"].max(0)
        out["position"][idx] = rs.uniform(lo, hi, (far, 3)).astype(np.float32)
    return out


@pytest.mark.parametrize("n,far,flags,keep", [(9, 0, 0, False), (9, 0, 0, True), (600, 20, b2r.FLAG_FORCE_BVH, False), (20000, 200, 0, False),
                                              (20000, 0, b2r.FLAG_REFERENCE_TREE, True)])
def test_refit_scene_equals_fresh_upload_and_oracle(n, far, flags, keep, hostcheck):
    """b2r_refit_scene (the drop-in for the rebuild-on-drag of Application.cpp:508-510): spheres move, the app rebuilds the reference BVH
    on the host (new leaf order; keep=True: it keeps the old one), the traversal tree keeps its topology and k_refit_level re-links its
    leaves and recomputes its boxes on the GPU. (1) The device tree equals the host twin (same shared routine) bit for bit; (2) the frame
    equals a fresh upload of the same arrays traced by BRUTE FORCE on the GPU, and — with the rebuilt order — the oracle's render of the
    moved scene (bit-exact on both pipelines, Q9 included); (3) the captured CUDA graph survives the
    edit; (4) the quality ratio is reported; (5) refitting back restores flatten_bvh's tree bit for bit."""
    import ctypes as C
    rs = np.random.RandomState(77 + n + far)
    sc = scenes.default_scene() if n == 9 else scenes.random_scene(n, light_every=40)
    w, h, mb = 160, 96, 8
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=2, flags=flags)
    r.Accumulate(2)                                     # graph captured on the unedited scene
    before_wide, _ = r.wide_nodes()
    prims_a = r.scene.prims.copy(); nodes_a = r.scene.nodes.copy(); ids_a = r.scene.prim_ids.copy()
    geo2 = _moved_geometry(sc["geometry"], rs, far=far)
    q = r.RefitScene(geo2, keep_order=keep); r.ResetAccumulator(); r.reset_counters(); r.Accumulate(4)
    got = r.buckets_host()
    prims_b = r.scene.prims.copy(); ids_b = r.scene.prim_ids.copy()
    assert keep == np.array_equal(ids_a, ids_b) or n == 9
    # (1) device tree == host twin
    wide, _ = r.wide_nodes(); obox = r.origin_box()   # the host twin sizes its leaves for the same origin box
    prim_of_geom_b = np.zeros(n, np.uint32); prim_of_geom_b[ids_b] = np.arange(n, dtype=np.uint32)
    remap = np.ascontiguousarray(prim_of_geom_b[ids_a])
    nw = C.c_uint32(0); cost = (C.c_double * 2)(); twin = np.zeros_like(wide)
    use_ref_tree = bool(flags & b2r.FLAG_REFERENCE_TREE)
    hostcheck.hc_refit(C.c_void_p(prims_a.ctypes.data), C.c_void_p(nodes_a.ctypes.data) if use_ref_tree else None, len(nodes_a) if use_ref_tree else 0,
                       C.c_void_p(prims_b.ctypes.data), C.c_void_p(remap.ctypes.data), n, C.c_void_p(twin.ctypes.data), C.byref(nw), cost, None, 0, None, None,
                       C.c_void_p(obox.ctypes.data))
    assert nw.value == len(wide) and wide.tobytes() == twin.tobytes()
    inner = before_wide[:, :, 6].view(np.int32) >= 0
    assert np.array_equal(inner, wide[:, :, 6].view(np.int32) >= 0) and np.array_equal(before_wide[:, :, 6].view(np.int32)[inner], wide[:, :, 6].view(np.int32)[inner])  # topology kept
    assert abs(q - cost[1] / cost[0]) <= 1e-5 * q
    print(f"refit n={n} far={far} keep_order={keep}: quality ratio {q:.4f}")
    if far: assert q > 1.0
    # (2a) fresh upload of the same arrays, brute force on the GPU
    sc2 = scenes.Scene(name="moved", geometry=geo2, material=sc["material"], camera=sc["camera"], ambient=sc["ambient"], hdri=None)
    ps2 = b2r.PreparedScene(sc2, w, h)
    if keep: ps2.prims = prims_b; ps2.prim_ids = ids_b
    else: assert all(np.array_equal(ps2.prims[k], prims_b[k]) for k in ("position", "radius_sq", "material_ID"))
    f = b2r.Renderer(ps2, w, h, max_bounces=mb, buckets=2, flags=b2r.FLAG_FORCE_BRUTE); f.Accumulate(4)
    fresh = f.buckets_host()
    frac = divergent_fraction(got, fresh)
    # (2b) the oracle on the moved scene (it rebuilds the reference BVH: the order the app gets after an edit)
    o = oracle_for(sc2, w, h, mb, 2); o.accumulate(4)
    frac_o = divergent_fraction(got, o.buckets())
    print(f"refit n={n}: divergent pixel fraction vs fresh brute-force upload {frac:.3e}, vs oracle {frac_o:.3e}")
    assert got.tobytes() == fresh.tobytes()
    if not keep:
        assert got.tobytes() == o.buckets().tobytes()
        gc, oc = r.counters(), o.counters()
        assert gc["extension_rays"] == oc["extension_rays"]
    # (5) back to the original spheres and order: the device tree is flatten_bvh's again, ratio 1
    q1 = r.RefitScene(sc["geometry"], keep_order=False)
    back, _ = r.wide_nodes()
    assert back.tobytes() == before_wide.tobytes() and abs(q1 - 1.0) < 1e-6
    r.close(); f.close()


def test_refit_scene_error_behaviour():
    sc = scenes.random_scene(300, light_every=40)
    r = b2r.Renderer(None, 64, 48)
    ps = b2r.PreparedScene(sc, 64, 48)
    import ctypes as C
    q = C.c_float(0)
    args = lambda p: (C.c_void_p(p.prims.ctypes.data), len(p.prims), C.c_void_p(p.material.ctypes.data), len(p.material), C.c_void_p(p.lights.ctypes.data), len(p.lights),
                      C.c_void_p(p.geometry.ctypes.data), len(p.geometry), C.byref(q))
    assert b2r.lib().b2r_refit_scene(r._h, *args(ps)) == b2r.ERR_STATE        # no topology yet
    r.SetScene(ps)
    assert b2r.lib().b2r_refit_scene(r._h, *args(ps)) == b2r.OK and abs(q.value - 1.0) < 1e-6
    other = b2r.PreparedScene(scenes.random_scene(301, light_every=40), 64, 48)
    assert b2r.lib().b2r_refit_scene(r._h, *args(other)) == b2r.ERR_ARG        # a refit keeps the sphere count
    bad = b2r.PreparedScene(sc, 64, 48); bad.prims = bad.prims.copy(); bad.prims["material_ID"][3] = 99
    assert b2r.lib().b2r_refit_scene(r._h, *args(bad)) == b2r.ERR_ARG
    r.close()


def test_team_mode_on_one_gpu_equals_plain_render():
    """b2r_team_* with a team of one: the same hand-shake kernels, slab resolve and copy paths as on N GPUs (the 2-GPU case is
    tests/test_multigpu_gpu.py), frames bit-identical to Render(); a resize while the team is open is refused."""
    import torch
    sc = scenes.default_scene()
    w, h = 256, 144
    a = b2r.Renderer(sc, w, h, max_bounces=8, buckets=8); b = b2r.Renderer(sc, w, h, max_bounces=8, buckets=8)
    b.team_open([b.team_export()], 0)
    pinned = torch.empty((h, w, 4), dtype=torch.float32, pin_memory=True).numpy()
    for k, n in enumerate((8, 16, 8)):
        a.ResetAccumulator(); a.Accumulate(n); assert a.Render()
        b.ResetAccumulator(); b.Accumulate(n)
        if k == 1:
            assert b.RenderTeam(out=pinned, use_async=True); b.WaitFrame(); got = pinned
        else:
            assert b.RenderTeam(); got = b.framebuffer
        assert got.tobytes() == a.framebuffer.tobytes()
    a.Accumulate(8); assert a.Render(); b.Accumulate(8); assert b.RenderTeam()      # progressive, no reset in between
    assert b.framebuffer.tobytes() == a.framebuffer.tobytes()
    b.Accumulate(3); assert not b.RenderTeam()                                      # accumulations % K != 0: no-op like Renderer::Render
    assert b.team_error() == 0
    with pytest.raises(b2r.B2RError):
        b.Resize(128, 64)
    b.team_close(); b.Resize(128, 64)
    a.close(); b.close()


def test_samples_traced_ahead_are_invisible_to_the_caller():
    """The drop-in's call pattern is one Accumulate() per application frame (Application.cpp:379). The library traces 2, 4, ... 16 samples
    ahead while nothing changes and folds them on the later calls. Bucket sums after every single call must be exactly those of a renderer
    that traces one sample per call (B2R_FLAG_NO_SPECULATION) and of one Accumulate(n) — including across a camera change, a reset, a
    jump of the sample index and a mixed Accumulate(1) / Accumulate(n) sequence, on both pipelines."""
    for sc, flags in ((scenes.default_scene(), 0), (scenes.random_scene(700, light_every=30), b2r.FLAG_FORCE_BVH)):
        w, h, K = 128, 80, 4
        a = b2r.Renderer(sc, w, h, max_bounces=6, buckets=K, flags=flags)
        b = b2r.Renderer(sc, w, h, max_bounces=6, buckets=K, flags=flags | b2r.FLAG_NO_SPECULATION)
        def both(fn):
            fn(a); fn(b)
        for i in range(21):                                   # 1, then batches of 2, 4, 8, 16 traced ahead
            both(lambda r: r.Accumulate(1))
            if i in (0, 1, 2, 5, 6, 13, 14, 20):
                assert a.buckets_host().tobytes() == b.buckets_host().tobytes(), i
        c = b2r.Renderer(sc, w, h, max_bounces=6, buckets=K, flags=flags); c.Accumulate(21)
        assert a.buckets_host().tobytes() == c.buckets_host().tobytes()
        cam2 = a.scene.camera.copy(); cam2[0] += 0.05                    # camera moves while samples traced ahead are pending: they are dropped
        both(lambda r: (r.SetCamera(cam2), r.ResetAccumulator()))
        for i in range(5):
            both(lambda r: r.Accumulate(1))
        assert a.buckets_host().tobytes() == b.buckets_host().tobytes()
        both(lambda r: r.Accumulate(6)); both(lambda r: r.Accumulate(1)); both(lambda r: r.Accumulate(1))   # mixed: pending samples are consumed in order
        assert a.buckets_host().tobytes() == b.buckets_host().tobytes()
        for r in (a, b): r.accumulations = 100                          # jump of the sample index (resume): pending samples no longer match
        for i in range(3):
            both(lambda r: r.Accumulate(1))
        assert a.buckets_host().tobytes() == b.buckets_host().tobytes() and a.accumulations == 103
        assert a.Render() == b.Render()
        assert a.framebuffer.tobytes() == b.framebuffer.tobytes()
        a.close(); b.close(); c.close()


def test_bucket_checkpoint_file_resumes_bit_identically(tmp_path):
    """b2r_save_checkpoint / b2r_load_checkpoint: 11 samples, save, a NEW renderer loads the file and goes on for 13 samples — bucket sums and
    frame equal 24 straight samples bit for bit (RNG streams are a function of the sample index, Q2-Q3); the file is refused for another
    configuration, when truncated and when a payload byte is flipped."""
    sc = scenes.random_scene(500, light_every=25)
    w, h, K, mb = 160, 96, 8, 6
    a = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K); a.Accumulate(11)
    path = tmp_path / "run.b2rk"; a.SaveCheckpoint(path); a.close()
    assert path.stat().st_size == 64 + K * 3 * w * h * 4
    b = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K); b.LoadCheckpoint(path)
    assert b.accumulations == 11
    b.Accumulate(13); assert b.Render()
    c = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K); c.Accumulate(24); assert c.Render()
    assert b.buckets_host().tobytes() == c.buckets_host().tobytes() and b.framebuffer.tobytes() == c.framebuffer.tobytes()
    for kw in (dict(max_bounces=mb + 1, buckets=K), dict(max_bounces=mb, buckets=K - 1), dict(max_bounces=mb, buckets=K, flags=b2r.FLAG_NO_MIS)):
        d = b2r.Renderer(sc, w, h, **kw)
        with pytest.raises(b2r.B2RError) as e: d.LoadCheckpoint(path)
        assert e.value.code == b2r.ERR_STATE
        d.close()
    raw = bytearray(path.read_bytes())
    (tmp_path / "short.b2rk").write_bytes(raw[:-4]); raw[1000] ^= 1; (tmp_path / "flipped.b2rk").write_bytes(raw); (tmp_path / "junk.b2rk").write_bytes(b"not a checkpoint" * 8)
    for name in ("short.b2rk", "flipped.b2rk", "junk.b2rk", "missing.b2rk"):
        with pytest.raises(b2r.B2RError) as e: b.LoadCheckpoint(tmp_path / name)
        assert e.value.code == b2r.ERR_ARG
    assert b.buckets_host().tobytes() == c.buckets_host().tobytes()   # a refused file leaves the renderer untouched
    b.close(); c.close()


@pytest.mark.parametrize("n", [5, 700, 20000])
def test_gpu_built_tree_equals_host_twin_and_brute_force(n, hostcheck):
    """B2R_FLAG_GPU_TREE: b2r_upload_scene builds the traversal tree on the device (Morton keys, CUB radix sort, implicit 4-ary links, refit
    passes). (1) The device tree equals the host twin build_packed_tree bit for bit; (2) the frame equals brute force on the GPU and the
    default SAH tree's; (3) a scene edit refits the device-built tree (leaf matching done lazily) and still equals brute force; (4) switching
    the flag off again uploads the SAH tree."""
    import ctypes as C
    sc = scenes.random_scene(n, light_every=20)
    w, h, mb = 160, 96, 8
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=2, flags=b2r.FLAG_FORCE_BVH | b2r.FLAG_GPU_TREE); r.Accumulate(4)
    wide, ms = r.wide_nodes(); obox = r.origin_box()
    nw = C.c_uint32(0); m2 = C.c_uint32(0); twin = np.zeros_like(wide)
    prims = np.ascontiguousarray(r.scene.prims)
    hostcheck.hc_packed_tree(C.c_void_p(prims.ctypes.data), n, C.c_void_p(obox.ctypes.data), C.c_void_p(twin.ctypes.data), C.byref(nw), C.byref(m2))
    assert nw.value == len(wide) and m2.value == ms and wide.tobytes() == twin.tobytes()
    got = r.buckets_host()
    b = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=2, flags=b2r.FLAG_FORCE_BRUTE); b.Accumulate(4)
    s = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=2, flags=b2r.FLAG_FORCE_BVH); s.Accumulate(4)
    assert got.tobytes() == b.buckets_host().tobytes() == s.buckets_host().tobytes()
    # (3) edit
    rs = np.random.RandomState(n)
    geo2 = _moved_geometry(sc["geometry"], rs, far=min(3, n // 2))
    q = r.RefitScene(geo2); r.ResetAccumulator(); r.Accumulate(4)
    sc2 = scenes.Scene(name="moved", geometry=geo2, material=sc["material"], camera=sc["camera"], ambient=sc["ambient"], hdri=None)
    b.SetScene(sc2); b.ResetAccumulator(); b.Accumulate(4)
    assert r.buckets_host().tobytes() == b.buckets_host().tobytes() and q > 0.0   # (the ratio can fall below 1: moved spheres may shrink the boxes)
    # (4) flag off: the next upload builds the SAH tree on the host again
    r.set_flags(b2r.FLAG_FORCE_BVH); r.SetScene(sc); r.ResetAccumulator(); r.Accumulate(4)
    wide2, _ = r.wide_nodes(); s_wide, _ = s.wide_nodes()
    assert r.buckets_host().tobytes() == got.tobytes() and wide2.shape == s_wide.shape
    r.close(); b.close(); s.close()


@pytest.mark.parametrize("three", [False, True])
@pytest.mark.parametrize("n", [2, 5, 6, 17, 700, 20000, 100000])
def test_gpu_sweep_tree_equals_host_twin_and_sah_tree_frame(n, three):
    """B2R_FLAG_GPU_TREE | B2R_FLAG_GPU_SAH: the device cuts the curve order top-down where the surface-area heuristic along the curve is
    smallest (k_sweep_*: segmented scans, an atomic minimum per run and round, one 4-byte read-back per level). The device tree equals the host
    twin build_sweep_tree bit for bit, and the frame rendered through it the default SAH tree's, also after a refit (tests/gpucheck/
    sweep_tree_check.py). three: B2R_FLAG_GPU_SAH3, the same sweep over the x, y and z orders at once (k_sweep3_*; twin build_sweep3_tree)."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpucheck"))
    import sweep_tree_check
    assert sweep_tree_check.check(n, three=three) if n < 100000 else sweep_tree_check.check(n, 320, 192, 1, three=three)   # (C3's scene: one sample of a larger frame)


def test_gpu_sweep_tree_falls_back_to_the_packed_tree_when_too_deep(hostcheck):
    """A hundred copies of one sphere: every cut of that run costs the same, the first is taken, so the sweep tree peels them off one by one
    and would be deeper than the traversal stack allows (the host twin gives up); the upload links the packed tree instead (device tree ==
    packed twin), the frame equals brute force, and the next scene gets its sweep tree again."""
    import ctypes as C
    sc = scenes.Scene(scenes.default_scene()); d = sc["geometry"]
    sc["geometry"] = np.ascontiguousarray(np.concatenate([d, np.repeat(d[3:4], 100)])); n = len(sc["geometry"])
    flags = b2r.FLAG_FORCE_BVH | b2r.FLAG_GPU_TREE | b2r.FLAG_GPU_SAH
    r = b2r.Renderer(sc, 96, 64, max_bounces=4, buckets=2, flags=flags); r.Accumulate(2)
    wide, ms = r.wide_nodes(); obox = r.origin_box(); prims = np.ascontiguousarray(r.scene.prims)
    nw = C.c_uint32(0); m2 = C.c_uint32(0)
    assert hostcheck.hc_sweep_tree(C.c_void_p(prims.ctypes.data), n, C.c_void_p(obox.ctypes.data), None, C.byref(nw), C.byref(m2)) == 1
    twin = np.zeros_like(wide)
    hostcheck.hc_packed_tree(C.c_void_p(prims.ctypes.data), n, C.c_void_p(obox.ctypes.data), C.c_void_p(twin.ctypes.data), C.byref(nw), C.byref(m2))
    assert nw.value == len(wide) and m2.value == ms and wide.tobytes() == twin.tobytes()
    b = b2r.Renderer(sc, 96, 64, max_bounces=4, buckets=2, flags=b2r.FLAG_FORCE_BRUTE); b.Accumulate(2)
    assert r.buckets_host().tobytes() == b.buckets_host().tobytes()
    sc2 = scenes.random_scene(300, light_every=20)
    r.SetScene(sc2); r.ResetAccumulator(); r.Accumulate(2); b.SetScene(sc2); b.ResetAccumulator(); b.Accumulate(2)
    assert r.buckets_host().tobytes() == b.buckets_host().tobytes()
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpucheck"))
    import sweep_tree_check
    assert len(r.wide_nodes()[0]) == sweep_tree_check.twin_nodes(np.ascontiguousarray(r.scene.prims), r.origin_box())
    r.close(); b.close()


def test_packet_traversal_of_camera_rays_equals_per_lane_walks():
    """k_intersect_packet walks the tree once per warp for the camera rays (bounce 0). Every lane's closest hit must be what its own walk
    gives: same bucket sums, bit for bit, as a context created with the per-lane kernel at bounce 0 (B2R_NO_PACKET, read at b2r_create),
    on a scene with many small spheres (lanes of one packet hit different spheres and miss), a wide-angle camera (divergent packets), a
    deep tree of nested spheres (the warp stack), and in reference-exact mode."""
    cases = [(scenes.random_scene(3000, light_every=25), 160, 96, 0), (scenes.random_scene(20000, light_every=40), 320, 192, b2r.FLAG_REFERENCE_EXACT)]
    wide = scenes.random_scene(3000, light_every=25); wide["camera"] = dict(wide["camera"]); wide["camera"]["focal_length"] = 6.0; cases.append((wide, 160, 96, 0))
    nested = scenes.Scene(scenes.default_scene()); n = 300
    geo = np.zeros(n, scenes.SPHERE_DTYPE); geo["radius_sq"] = (np.linspace(0.01, 1.2, n) ** 2).astype(np.float32); geo["position"][:, 0] = 0.3; geo["material_ID"] = np.arange(n) % 9
    nested["geometry"] = geo; cases.append((nested, 160, 96, b2r.FLAG_FORCE_BVH))
    for sc, w, h, flags in cases:
        a = b2r.Renderer(sc, w, h, max_bounces=6, buckets=2, flags=flags | b2r.FLAG_FORCE_BVH); a.Accumulate(4)
        os.environ["B2R_NO_PACKET"] = "1"
        try:
            b = b2r.Renderer(sc, w, h, max_bounces=6, buckets=2, flags=flags | b2r.FLAG_FORCE_BVH)
        finally:
            del os.environ["B2R_NO_PACKET"]
        b.Accumulate(4)
        assert a.buckets_host().tobytes() == b.buckets_host().tobytes()
        ca, cb = a.counters(), b.counters()
        assert ca["extension_rays"] == cb["extension_rays"] and ca["shadow_rays"] == cb["shadow_rays"] and ca["shaded_hits"] == cb["shaded_hits"]
        a.close(); b.close()
