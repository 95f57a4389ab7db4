"""The oracle against THE REFERENCE ITSELF: Renderer<>::Accumulate / Render (Renderer.hpp with DataStreams.hpp, BVH.hpp, Scene.hpp,
Camera.hpp, Sampling.hpp, ...) compiled from /root/reference into oracle/_ref/librefrenderer.so by oracle/ref_renderer_build.sh.

The oracle's slot-exact mode (flag ORC_SLOT_EXACT: closest-hit SIMD blocks of 8 + scalar tail by stream slot, BVH.hpp:250-286) must
reproduce the reference's five bucket-sum planes and its tonemapped RGBA32F frame BIT FOR BIT; the oracle's canonical mode (the
SIMD-FMA sphere formula for every ray — what the GPU computes, DESIGN.md "Numerics") must stay within north_star's tolerance of it
(per-sample radiance within 1e-4 relative except a small, reported fraction of divergent paths; converged RMSE < 1e-3).

* tests/golden/renderer_kat.json holds the reference's outputs (tests/gen_golden.py) and travels everywhere;
* where the library is present (build container; GPU box, to which oracle/_ref/ is shipped) the comparison also runs live."""
import hashlib
import json
import os

import numpy as np
import pytest

import gen_golden
import oracle_py
import scenes

G = os.path.join(os.path.dirname(__file__), "golden")
live = pytest.mark.skipif(not oracle_py.have_reference_renderer(), reason="oracle/_ref/librefrenderer.so not present (built only where /root/reference exists)")


def oracle_run(sc, w, h, mb, n, first, flags):
    o = oracle_py.Oracle(w, h, max_bounces=mb, K=5, flags=flags); o.set_scene(sc)
    if first:
        o.set_accumulations(first)
    o.accumulate(n, threads=1)
    rc, frame = o.render()  # rc 0 = resolved, 1 = no-op (accumulations % K != 0)
    b = o.buckets(); o.close()
    return b, rc == 0, frame


def test_oracle_slot_exact_mode_reproduces_reference_renderer_golden():
    want = json.load(open(os.path.join(G, "renderer_kat.json")))
    for name, sc, w, h, mb, n, first in gen_golden.renderer_cases():
        b, acted, frame = oracle_run(sc, w, h, mb, n, first, oracle_py.ORC_SLOT_EXACT)
        got = gen_golden.renderer_record(b, acted, frame)
        assert got["sha256_buckets"] == want[name]["sha256_buckets"], f"{name}: bucket sums differ from the reference's Renderer::Accumulate"
        assert got["render_acted"] == want[name]["render_acted"] and got["sha256_frame"] == want[name]["sha256_frame"], f"{name}: frame differs from Renderer::Render"


@live
@pytest.mark.parametrize("threads", ["1", "4"])
def test_live_bit_exact_and_schedule_independent(threads, monkeypatch):
    """fresh cases (not in the fixture), and the reference's tile fan-out on 1 and 4 threads gives the same bits"""
    monkeypatch.setenv("REF_THREADS", threads)
    cases = [("default", scenes.default_scene(), 112, 80, 8, 15, 0), ("random900", scenes.random_scene(900, light_every=30, seed=77), 64, 64, 16, 5, 5),
             ("sky", scenes.bvh_test_scene(64, hdri=scenes.synthetic_hdri(32, 16, seed=9)), 48, 48, 4, 10, 0),
             ("brdf_test", scenes.brdf_test_scene(hdri=scenes.synthetic_hdri(24, 12, seed=2)), 64, 48, 8, 10, 0)]  # Application.cpp:123-217: albedo-0 spheres, q = 1 roulette
    for name, sc, w, h, mb, n, first in cases:
        r = oracle_py.ReferenceRenderer(sc, w, h, mb)
        if first:
            r.set_accumulations(first)
        r.accumulate(n); rb = r.buckets(); racted, rframe = r.render(); r.close()
        b, acted, frame = oracle_run(sc, w, h, mb, n, first, oracle_py.ORC_SLOT_EXACT)
        assert rb.tobytes() == b.tobytes(), name
        assert racted == acted and rframe.tobytes() == frame.tobytes(), name


def test_canonical_mode_within_north_star_tolerance_of_reference():
    """What the GPU computes (SIMD-FMA formula for every closest-hit ray) against the reference: divergent-path fraction and RMSE. The
    reference's side — its first sample (bucket 1) and its 200-spp frame of this render — is tests/golden/reference_default_160x96_mb16.npz
    (tests/gen_golden.py)."""
    sc = scenes.default_scene(); w, h, mb = 160, 96, 16
    ref = np.load(os.path.join(G, "reference_default_160x96_mb16.npz")); one, rframe = ref["first_sample"], ref["frame_200spp"]  # sample index 1 lands in bucket 1 (Q1)
    o = oracle_py.Oracle(w, h, max_bounces=mb, K=5); o.set_scene(sc); o.accumulate(1, threads=1); mine = o.buckets()[1].copy()
    o.accumulate(199); rc, frame = o.render(); acted = rc == 0; o.close()
    rel = np.abs(mine - one) / np.maximum(np.abs(one), 1e-6)
    divergent = float((rel > 1e-4).any(axis=0).mean())
    rmse = float(np.sqrt(np.mean((frame[..., :3] - rframe[..., :3]) ** 2)))
    print(f"canonical oracle vs reference renderer: divergent per-sample pixel fraction {divergent:.3e}, converged (200 spp) tonemapped RMSE {rmse:.3e}")
    assert acted and divergent < 2e-3 and rmse < 1e-3


# ---------------------------------------------------------------------------------------------- GGX closure (the reference's `#define BRDF 1` build)
live_ggx = pytest.mark.skipif(not oracle_py.have_reference_renderer(ggx=True), reason="oracle/_ref/librefrenderer_ggx.so not present (built only where /root/reference exists)")


def test_oracle_ggx_mode_reproduces_the_references_brdf1_build_golden():
    """ORC_GGX restates Closure<GGX> (DataStreams.hpp:184-219) and Sampling.hpp:249-309; the fixture holds what the reference's own
    Renderer<> computes when built with `#define BRDF 1` (and the all-zero gloss_decay_table that build needs to compile at all)."""
    want = json.load(open(os.path.join(G, "renderer_ggx_kat.json")))
    for name, sc, w, h, mb, n, first in gen_golden.renderer_ggx_cases():
        b, acted, frame = oracle_run(sc, w, h, mb, n, first, oracle_py.ORC_SLOT_EXACT | oracle_py.ORC_GGX)
        got = gen_golden.renderer_record(b, acted, frame)
        assert got["sha256_buckets"] == want[name]["sha256_buckets"], f"{name}: bucket sums differ from the reference's BRDF 1 build"
        assert got["render_acted"] == want[name]["render_acted"] and got["sha256_frame"] == want[name]["sha256_frame"], name
        assert np.isfinite(b).all()


@live_ggx
def test_live_ggx_bit_exact():
    cases = [("default", scenes.default_scene(), 112, 80, 8, 10, 0), ("ggx_random900", scenes.ggx_random_scene(900, light_every=30), 64, 64, 16, 5, 5),
             ("brdf_test", scenes.brdf_test_scene(hdri=scenes.synthetic_hdri(24, 12, seed=2)), 64, 48, 4, 10, 0)]
    for name, sc, w, h, mb, n, first in cases:
        r = oracle_py.ReferenceRenderer(sc, w, h, mb, ggx=True)
        if first:
            r.set_accumulations(first)
        r.accumulate(n); rb = r.buckets(); racted, rframe = r.render(); r.close()
        b, acted, frame = oracle_run(sc, w, h, mb, n, first, oracle_py.ORC_SLOT_EXACT | oracle_py.ORC_GGX)
        assert rb.tobytes() == b.tobytes(), name
        assert racted == acted and rframe.tobytes() == frame.tobytes(), name
        # and it is a different image from the Lambertian build's (the closure is really in use)
        lb, _, _ = oracle_run(sc, w, h, mb, n, first, oracle_py.ORC_SLOT_EXACT)
        assert lb.tobytes() != b.tobytes(), name
