"""Thin-lens depth of field (b2r_set_lens): the camera ray leaves a point L of a lens disk of radius R and passes through the point where the
pinhole ray of the same pixel sample meets the focus plane z = -F (b2r_math.h camera_lens_ray). The reference computes an aperture it never
uses (SURVEY Q22), so there is no reference result: the routine is pinned bit for bit to the oracle's restatement (oracle.cpp
generate_ray_lens), its geometry is checked in float64, and every kernel that makes camera rays is pinned to the oracle and to brute force.
R = 0 is the pinhole camera through the existing kernel instantiations, bit for bit.

The lens restatement lives in tests/lenscheck/lens_oracle.cpp: the oracle (oracle/oracle.cpp) compiled with a thin-lens camera ray, so
frames rendered by the oracle with a lens are available without changing the oracle itself; tests/lenscheck/lens_taps.cpp runs the kernels'
camera routines on the host. This module compiles both (g++, the oracle's flags) into a temporary directory.

CPU tier: the routine on the host against the oracle, geometry, the lens RNG stream, oracle frames and depth-of-field sanity. GPU tier
(-m gpu): everything the kernels do with a lens."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import b2r
import oracle_py
import scenes
from conftest import have_gpu
from test_traversal_exact import TREE_FLAGS, _declare, _scene_of
from test_traversal_kernels import PACKET_SCENES, _grazing_packet_scene, _packet_scene, brute_closest, differ

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G = os.path.join(HERE, "golden")
needs_gpu = pytest.mark.skipif(not have_gpu(), reason="needs a CUDA device")
f32 = np.float32


_LENSCHECK = None


def lenscheck():
    """tests/lenscheck compiled once per session into a temporary directory: the oracle with a lens (lo_*, orc_*) and the kernels' camera
    routines on the host (hc_lens_ray, hc_primary_rays)"""
    global _LENSCHECK
    if _LENSCHECK is None:
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_lenscheck_"), "liblenscheck.so")
        src = os.path.join(HERE, "lenscheck")
        subprocess.check_call(["g++", "-std=c++17", "-fPIC", "-shared", "-pthread", "-fno-fast-math", "-O2", "-mavx2", "-mfma", "-ffp-contract=off",
                               "-I", os.path.join(ROOT, "oracle"), "-I", os.path.join(ROOT, "cpu-raytracing-experiments_b200", "csrc"), "-I/usr/local/cuda/include",
                               os.path.join(src, "lens_oracle.cpp"), os.path.join(src, "lens_taps.cpp"), "-o", out])
        L = C.CDLL(out)
        ref = oracle_py.lib()
        for name in ("orc_create", "orc_destroy", "orc_set_scene", "orc_set_camera_lookat", "orc_set_camera_raw", "orc_get_camera_raw", "orc_reset",
                     "orc_set_accumulations", "orc_accumulate", "orc_read_buckets", "orc_render", "orc_read_counters", "orc_reset_counters", "orc_trace_closest"):
            fn, r = getattr(L, name), getattr(ref, name); fn.argtypes = r.argtypes; fn.restype = r.restype
        vp, f, i32, u32 = C.c_void_p, C.c_float, C.c_int32, C.c_uint32
        L.lo_set_lens.argtypes = [vp, f, f]; L.lo_set_lens.restype = None
        L.lo_generate_lens_ray_at.argtypes = [vp, i32, i32, vp, vp, vp]; L.lo_generate_lens_ray_at.restype = None
        L.lo_generate_rays.argtypes = [vp, u32, vp]; L.lo_generate_rays.restype = None
        L.hc_lens_ray.argtypes = [vp, i32, i32, vp, f, f, vp, vp]; L.hc_lens_ray.restype = None
        L.hc_primary_rays.argtypes = [vp, u32, u32, u32, u32, f, f, vp]; L.hc_primary_rays.restype = None
        _LENSCHECK = L
    return _LENSCHECK


class LensOracle(oracle_py.Oracle):
    """oracle_py.Oracle on the oracle compiled with a thin lens (tests/lenscheck/lens_oracle.cpp); set_lens(0, F) or no call = the pinhole"""

    def __init__(self, width, height, max_bounces=16, K=5, flags=0):
        self.L = lenscheck()
        self.h = self.L.orc_create(width, height, max_bounces, K, flags)
        assert self.h
        self.width, self.height, self.K, self.max_bounces = width, height, K, max_bounces
        self.npix = width * height
        self.L.lo_set_lens(self.h, 0.0, 1.0)

    def set_lens(self, radius, focus_distance):
        self.L.lo_set_lens(self.h, radius, focus_distance)

    def generate_rays(self, acc):
        out = np.empty((self.npix, 6), np.float32); self.L.lo_generate_rays(self.h, acc, _p(out)); return out


@pytest.fixture(scope="module")
def hc(hostcheck):
    return _declare(hostcheck)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _unit_quat(rs):
    q = rs.randn(4); return (q / np.linalg.norm(q)).astype(np.float32)


def _rot(q, v):
    """rotate v (n, 3) by the unit quaternion q = (w, x, y, z), float64"""
    w, x, y, z = (float(c) for c in q)
    n = w * w + x * x + y * y + z * z; w, x, y, z = w / np.sqrt(n), x / np.sqrt(n), y / np.sqrt(n), z / np.sqrt(n)
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                  [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                  [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    return np.asarray(v, np.float64) @ R.T


def _cameras(seed=21):
    """(cam11, R, F): look-at cameras (as b2r_camera_lookat makes them) and raw random orientations; tiny and huge F, R far beyond the scene"""
    rs = np.random.RandomState(seed); out = []
    for k in range(24):
        if k % 2 == 0:
            cam = b2r.camera_lookat(rs.uniform(-50, 50, 3), rs.randn(3), 64, 48, float(rs.uniform(10, 80)))
        else:
            cam = np.r_[rs.uniform(-1e3, 1e3, 3), _unit_quat(rs), 32.0, 24.0, -rs.uniform(10, 500), 1.0].astype(np.float32)
        R = [0.05, 1.0, 20.0, 1e4][k % 4]
        F = [1e-3, 3.0, 150.0, 1e6][(k // 4) % 4]
        out.append((cam, f32(R), f32(F)))
    return out


def _oracle_raw(cam, w=64, h=48, mb=16):
    o = LensOracle(w, h, max_bounces=mb, K=1)
    o.L.orc_set_camera_raw(o.h, _fp(np.ascontiguousarray(cam[0:3])), _fp(np.ascontiguousarray(cam[3:7])), float(cam[7]), float(cam[8]), float(cam[9]), float(cam[10]))
    return o


def _sample_grid(rs, n):
    s = rs.uniform(0, 1, (n, 4)).astype(np.float32)
    s[:8] = np.array([[0, 0, 0, 0], [1, 1, 1, 1], [0, 1, 1, 0], [1, 0, 0, 1], [0.5, 0.5, 1, 1], [0, 0, 1, 0.25], [1, 1, 0, 0.75], [0.999, 0.001, 1, 0.5]], np.float32)
    return s


# ------------------------------------------------------------------------------------------------ CPU tier
def test_lens_routine_bit_exact_with_the_oracle():
    """camera_lens_ray (the kernels' routine, on the host) == the lens oracle's generate_ray_lens, bit for bit: random and rotated cameras, samples
    at 0 and 1.0 (next_unit can return 1, Q4), F from 1e-3 to 1e6, R from 0.05 to 1e4 (far larger than the scene)."""
    rs = np.random.RandomState(22); n_bad = 0; n = 0
    for cam, R, F in _cameras():
        o = _oracle_raw(cam); o.set_lens(R, F)
        for s in _sample_grid(rs, 40):
            x, y = int(rs.randint(0, 64)), int(rs.randint(0, 48))
            a = np.zeros(6, np.float32); b = np.zeros(6, np.float32); px, ln = s[:2].copy(), s[2:].copy()   # (named: a temporary's buffer may be reused)
            lenscheck().hc_lens_ray(_p(cam), x, y, _p(px), R, F, _p(ln), _p(a))
            o.L.lo_generate_lens_ray_at(o.h, x, y, _p(px), _p(ln), _p(b))
            n_bad += int(a.tobytes() != b.tobytes()); n += 1
        o.close()
    assert n_bad == 0, f"{n_bad} of {n} rays differ"


def test_primary_rays_and_lens_stream_bit_exact_with_the_oracle():
    """primary_path<LENS> (the camera rays every kernel makes, with the lens sample drawn from branch 2 * max_bounces) == the oracle's
    generate_rays with a lens, for every pixel and several sample indices; R = 0 takes the pinhole path of both."""
    for cam, R, F in _cameras(23)[:6]:
        for mb in (1, 4, 16):
            o = _oracle_raw(cam, 64, 48, mb); o.set_lens(R, F)
            for acc in (1, 2, 77):
                mine = np.empty((64 * 48, 6), np.float32)
                lenscheck().hc_primary_rays(_p(cam), 64, 48, mb, acc, R, F, _p(mine))
                assert mine.tobytes() == o.generate_rays(acc).tobytes(), (mb, acc)
            o.set_lens(0.0, F)
            mine = np.empty((64 * 48, 6), np.float32); lenscheck().hc_primary_rays(_p(cam), 64, 48, mb, 5, 0.0, F, _p(mine))
            assert mine.tobytes() == o.generate_rays(5).tobytes()
            o.close()


def test_lens_ray_geometry_in_float64():
    """Every origin lies in the lens plane within R (1 + 1e-6) of the eye (plus one rounding of the float sum pos + orient * L); every ray passes through its pixel's pinhole focus point
    pos + orient * (v * -F / z), to a relative 1e-5 of its distance from the origin (the rounding of the float origin, a few ulp of |pos|,
    moves the ray sideways by as much: it is allowed for)."""
    rs = np.random.RandomState(24)
    worst_r, worst_plane, worst_focus = 0.0, 0.0, 0.0
    for cam, R, F in _cameras(25):
        pos, q = cam[0:3].astype(np.float64), cam[3:7]
        for s in _sample_grid(rs, 30):
            x, y = int(rs.randint(0, 64)), int(rs.randint(0, 48))
            a = np.zeros(6, np.float32); px, ln = s[:2].copy(), s[2:].copy()
            lenscheck().hc_lens_ray(_p(cam), x, y, _p(px), R, F, _p(ln), _p(a))
            o, d = a[:3].astype(np.float64), a[3:].astype(np.float64)
            local = _rot(np.r_[q[0], -q[1:]], (o - pos)[None])[0]   # back into camera space
            worst_r = max(worst_r, np.linalg.norm(o - pos) / (R * (1 + 1e-6) + np.sqrt(3) * 2.0 ** -23 * np.abs(pos).max()))   # + the rounding of pos + orient * L
            worst_plane = max(worst_plane, abs(local[2]) / (1e-6 * float(R) + 4 * 2.0 ** -23 * np.abs(pos).max()))
            v = np.array([x + float(s[0]) - float(cam[7]), y + float(s[1]) - float(cam[8]), float(cam[9])])
            P = pos + _rot(q, (v * (-float(F) / float(cam[9])))[None])[0]
            t = np.dot(P - o, d) / np.dot(d, d)
            miss = np.linalg.norm(o + t * d - P) / (np.linalg.norm(P - o) + 2 * np.sqrt(3) * 2.0 ** -23 * np.abs(pos).max() / 1e-5)
            worst_focus = max(worst_focus, miss)
    assert worst_r <= 1.0 + 1e-6, worst_r
    assert worst_plane <= 1.0, worst_plane
    assert worst_focus <= 1e-5, worst_focus


@pytest.mark.parametrize("w,h,mb", [(1920, 1088, 16), (256, 144, 4), (64, 48, 1), (3840, 2160, 64)])
def test_lens_stream_is_used_by_nothing_else(w, h, mb):
    """The lens stream of pixel t is branch 2 mb of its seed range: seed(t) + 2 mb with seed(t) = t (2 mb + 1) (uint32, wrapping). The
    branches of all pixels of the frame that light samples (2b) and BRDF continuations (2b + 1) use, [seed(t), seed(t) + 2 mb), never hold it."""
    t = np.arange(w * h, dtype=np.uint64)
    seed = (t * np.uint64(2 * mb + 1)) & np.uint64(0xffffffff)
    lens = (seed + np.uint64(2 * mb)) & np.uint64(0xffffffff)
    used = ((seed[:, None] + np.arange(2 * mb, dtype=np.uint64)[None]) & np.uint64(0xffffffff)).ravel() if w * h * 2 * mb <= 1 << 26 else None
    if used is not None:
        assert np.intersect1d(lens, used).size == 0
    else:   # too many to list: below 2^32 nothing wraps, and every used value is != 2 mb (mod 2 mb + 1)
        assert int(seed[-1]) + 2 * mb < 2 ** 32
        assert (lens % np.uint64(2 * mb + 1) == np.uint64(2 * mb)).all()
    assert np.unique(lens).size == lens.size


def test_oracle_frames_pinhole_and_white_furnace():
    """R = 0 is the pinhole: an oracle that set a zero lens renders the bits of one that never set a lens. The white furnace with a lens
    still gives exactly ambient x texel at every pixel (the lens moves rays, it does not change what a closed sky returns)."""
    sc = scenes.default_scene()
    a = oracle_py.Oracle(128, 80, max_bounces=8, K=1); a.set_scene(sc); a.accumulate(2)
    b = LensOracle(128, 80, max_bounces=8, K=1); b.set_scene(sc); b.set_lens(0.0, 5.0); b.accumulate(2)
    c = LensOracle(128, 80, max_bounces=8, K=1); c.set_scene(sc); c.set_lens(0.3, 5.0); c.accumulate(2)
    assert a.buckets().tobytes() == b.buckets().tobytes()
    assert a.buckets().tobytes() != c.buckets().tobytes()
    wf = scenes.white_furnace()
    o = LensOracle(64, 48, max_bounces=16, K=1); o.set_scene(wf); o.set_lens(0.4, 2.0); o.accumulate(3)
    assert o.counters()["dropped"] == 0 and np.all(o.buckets()[0] == 3.0)


def _coverage(sphere_pos, radius, R, F, n_samples=64, w=128, h=128, z=-128.0):
    """fraction of the camera rays of n_samples sample indices that hit one sphere, per pixel (raster), camera at 0 looking down -z"""
    g = np.zeros(1, scenes.SPHERE_DTYPE); g["position"] = sphere_pos; g["radius_sq"] = f32(radius * radius)
    o = LensOracle(w, h, max_bounces=4, K=1); o.set_scene(_scene_of(g))
    cam = np.array([0, 0, 0, 1, 0, 0, 0, w / 2, h / 2, z, 1], np.float32)
    o.L.orc_set_camera_raw(o.h, _fp(cam[0:3].copy()), _fp(cam[3:7].copy()), float(cam[7]), float(cam[8]), float(cam[9]), 1.0)
    o.set_lens(R, F)
    hits = np.zeros(w * h)
    for acc in range(1, n_samples + 1):
        _, p = o.trace_closest(o.generate_rays(acc)); hits += p >= 0
    o.close()
    return oracle_py.tile_to_raster(hits / n_samples, w, h)


def _edge_band(profile, lo=0.1, hi=0.9):
    """width in pixels between the crossings of lo and hi on the rising (left) edge of a coverage profile, linearly interpolated"""
    def cross(level):
        i = int(np.argmax(profile >= level)); return i - 1 + (level - profile[i - 1]) / (profile[i] - profile[i - 1])
    return cross(hi) - cross(lo)


def test_depth_of_field_sanity():
    """A sphere on the focus plane covers the pinhole's pixels (to within one pixel of its silhouette); a sphere at 2F shows a partial
    coverage band across its silhouette edge whose width matches the analytic circle of confusion 2 R |z| |d - F| / (d F) pixels within 20 %
    (the 10 %-90 % width of a disk-blurred edge is measured and converted to the disk's diameter)."""
    F, R, z = 10.0, 1.0, 128.0
    pin = _coverage((0, 0, -F), 1.0, 0.0, F) >= 0.5
    lens = _coverage((0, 0, -F), 1.0, R, F) >= 0.5
    edge = np.zeros_like(pin)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            edge |= pin != np.roll(np.roll(pin, dy, 0), dx, 1)
    near_edge = edge.copy()
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            near_edge |= np.roll(np.roll(edge, dy, 0), dx, 1)
    assert pin.sum() > 100 and not ((pin != lens) & ~near_edge).any()
    d, r = 2 * F, 4.0
    cov = _coverage((0, 0, -d), r, R, F, n_samples=128)
    d_sil = d - r * r / d                                   # depth of the silhouette circle
    coc = 2 * R * z * abs(d_sil - F) / (d_sil * F)
    prof = cov[64, :].astype(np.float64)
    partial = ((prof > 0.02) & (prof < 0.98)).sum() / 2     # per edge
    assert partial >= 0.6 * coc, (partial, coc)
    rs = np.random.RandomState(26); m = 400000           # 10-90 width of a disk of diameter 1 blurring an edge, with the pixel's 1-pixel jitter
    rr, ph = np.sqrt(rs.uniform(0, 1, m)), rs.uniform(0, 2 * np.pi, m)
    spread = np.sort(0.5 * coc * rr * np.cos(ph) + rs.uniform(-0.5, 0.5, m))
    expect = spread[int(0.9 * m)] - spread[int(0.1 * m)]
    got = _edge_band(prof)
    assert abs(got / expect - 1.0) <= 0.2, (got, expect, coc)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@needs_gpu
def test_gpu_pinhole_untouched():
    """Both pipelines: no SetLens, SetLens(0, F), and a lens switched on then back to 0 give the same bucket sums and the committed golden digests."""
    g = json.load(open(os.path.join(G, "oracle_frames.json")))
    sc = scenes.default_scene(); sc2 = scenes.random_scene(2000, light_every=50)
    cases = [(sc, 320, 192, dict(max_bounces=8, buckets=5), 5, g["default_320x192_mb8_K5_acc5"]["sha256_buckets"]),
             (sc2, 160, 96, dict(max_bounces=8, buckets=1, flags=b2r.FLAG_FORCE_BRUTE), 1, g["random2000_160x96_mb8_K1_acc1"]["sha256_buckets"]),
             (sc2, 160, 96, dict(max_bounces=8, buckets=1, flags=b2r.FLAG_FORCE_BVH), 1, g["random2000_160x96_mb8_K1_acc1"]["sha256_buckets"])]
    for scene, w, h, kw, n, want in cases:
        for calls in [(), ((0.0, 7.0),), ((0.5, 7.0), (0.0, 7.0))]:
            r = b2r.Renderer(scene, w, h, **kw)
            for c in calls: r.SetLens(*c)
            r.Accumulate(n)
            got = hashlib.sha256(r.buckets_host().tobytes()).hexdigest(); r.close()
            assert got == want, (kw, calls)
        r = b2r.Renderer(scene, w, h, **kw)   # lens on after a pinhole frame, then off again: the graph is re-captured both times
        r.Accumulate(n); r.SetLens(0.5, 7.0); r.Accumulate(n); r.SetLens(0.0, 7.0); r.ResetAccumulator(); r.Accumulate(n)
        got = hashlib.sha256(r.buckets_host().tobytes()).hexdigest(); r.close()
        assert got == want, (kw, "on/off")


def _oracle_for(sc, w, h, mb, K, flags=0):
    o = LensOracle(w, h, max_bounces=mb, K=K, flags=flags); o.set_scene(sc); return o


@pytest.mark.gpu
@needs_gpu
def test_gpu_generate_rays_equal_the_oracle():
    """b2r_generate_rays with a lens == the oracle's generate_rays, every pixel, several sample indices and cameras."""
    rs = np.random.RandomState(27)
    for k in range(4):
        sc = scenes.default_scene(); sc["camera"] = dict(eye=tuple(rs.uniform(-20, 20, 3)), dir=tuple(rs.randn(3)), focal_length=float(rs.uniform(15, 60)), exposure=1.0)
        r = b2r.Renderer(sc, 96, 64, max_bounces=[1, 4, 8, 16][k], buckets=1)
        o = _oracle_for(sc, 96, 64, [1, 4, 8, 16][k], 1)
        R, F = [0.01, 0.3, 5.0, 200.0][k], [0.5, 8.0, 30.0, 1e4][k]
        r.SetLens(R, F); o.set_lens(R, F)
        for acc in (1, 3, 1000):
            assert r.generate_rays(acc).tobytes() == o.generate_rays(acc).tobytes(), (k, acc)
        r.close(); o.close()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("variant", ["lambertian", "ggx", "no_mis", "mb16", "count"])
def test_gpu_brute_pipeline_equals_the_oracle(variant):
    """k_bounce_brute's lens instantiations (per-ray sphere tests, the camera ray regenerated in the shading phase): bucket sums and the
    tonemapped frame bit for bit against the oracle."""
    sc = scenes.default_scene(); w, h, K = 192, 112, 2
    mb = 16 if variant == "mb16" else 8
    flags = {"ggx": b2r.FLAG_GGX, "no_mis": b2r.FLAG_NO_MIS, "count": b2r.FLAG_COUNT_TESTS}.get(variant, 0)
    oflags = {"ggx": oracle_py.ORC_GGX, "no_mis": oracle_py.ORC_NO_MIS}.get(variant, 0)
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=K, flags=flags | b2r.FLAG_FORCE_BRUTE)
    o = _oracle_for(sc, w, h, mb, K, oflags)
    r.SetLens(0.35, 4.5); o.set_lens(0.35, 4.5)
    r.Accumulate(4); o.accumulate(4)
    assert r.buckets_host().tobytes() == o.buckets().tobytes()
    assert r.Render(); rc, ref = o.render()
    assert r.framebuffer.tobytes() == ref.tobytes()
    r.close(); o.close()


C3_SMALL = dict(w=256, h=144, n=2)


@pytest.fixture(scope="module")
def c3_scene():
    return scenes.random_scene(100000)


def _c3_lens(sc):
    eye = np.asarray(sc["camera"]["eye"], np.float64)
    return 2.0, float(np.linalg.norm(eye))   # focused near the scene centre


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("tree", list(TREE_FLAGS) + ["refit", "no_packet"])
def test_gpu_bvh_pipeline_equals_brute_force(c3_scene, tree, monkeypatch):
    """C3's scene at 256x144, 2 samples, with a lens: the BVH kernels (packet kernel at bounce 0, or k_generate + the per-lane walk with
    B2R_NO_PACKET set before the context exists) equal a FORCE_BRUTE context bit for bit, for every tree flag and after a refit."""
    if tree == "no_packet": monkeypatch.setenv("B2R_NO_PACKET", "1")
    else: monkeypatch.delenv("B2R_NO_PACKET", raising=False)
    sc = c3_scene; R, F = _c3_lens(sc); w, h, n = C3_SMALL["w"], C3_SMALL["h"], C3_SMALL["n"]
    ref = b2r.Renderer(sc, w, h, max_bounces=6, buckets=1, flags=b2r.FLAG_FORCE_BRUTE); ref.SetLens(R, F); ref.Accumulate(n)
    want = ref.buckets_host(); ref.close()
    r = b2r.Renderer(sc, w, h, max_bounces=6, buckets=1, flags=b2r.FLAG_FORCE_BVH | TREE_FLAGS.get(tree, 0))
    if tree == "refit":
        geo = np.ascontiguousarray(sc["geometry"]).copy(); geo["position"][:, 1] += f32(0.5); r.RefitScene(geo); r.RefitScene(sc["geometry"])
    r.SetLens(R, F); r.Accumulate(n)
    got = r.buckets_host(); r.close()
    assert float(want.max()) > 0.0
    assert got.tobytes() == want.tobytes()


@pytest.mark.gpu
@needs_gpu
def test_gpu_bvh_pipeline_equals_the_oracle():
    sc = scenes.random_scene(2000, light_every=50); w, h = 160, 96
    r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=1, flags=b2r.FLAG_FORCE_BVH); o = _oracle_for(sc, w, h, 8, 1)
    eye = np.asarray(sc["camera"]["eye"], np.float64); R, F = 1.5, float(np.linalg.norm(eye))
    r.SetLens(R, F); o.set_lens(R, F); r.Accumulate(2); o.accumulate(2)
    assert r.buckets_host().tobytes() == o.buckets().tobytes()
    r.close(); o.close()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("name", ["edge_of_scene"] + PACKET_SCENES)
def test_gpu_packet_kernel_with_a_lens_equals_brute_force(hc, name):
    """k_intersect_packet's lens instantiation == hc_closest_brute over b2r_generate_rays, exactly: a camera at the edge of the scene with R
    larger than the origin box's slack, and the scenes test_traversal_kernels.py aims at the packet kernel (lens radius a few percent of the
    camera's distance to the scene, focused there)."""
    if name == "edge_of_scene":
        sc = scenes.random_scene(3000, light_every=40); lo = sc["geometry"]["position"].min(0); hi = sc["geometry"]["position"].max(0)
        eye = (float(hi[0]), float(hi[1]), float(hi[2]) + 1.0)
        sc["camera"] = dict(eye=eye, dir=(-1, -0.5, -1), focal_length=20.0, exposure=1.0)
        w = h = 64; accs = [1, 9]; R, F = 2.0 * float((hi - lo).max()), 50.0
    else:
        sc, w, h, accs = _packet_scene(name, hc)
        eye = np.asarray(sc["camera"]["eye"], np.float64)
        F = float(np.linalg.norm(sc["geometry"]["position"].astype(np.float64).mean(0) - eye)) or 1.0
        R = 0.02 * F
    r = b2r.Renderer(sc, w, h, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    if name == "grazing":   # spheres placed on this renderer's lens rays
        r.SetLens(R, F)
        g = _scene_of(_grazing_packet_scene(hc, r, accs[0])); g["camera"] = sc["camera"]; r.SetScene(g)
    r.SetLens(R, F)
    box = r.origin_box(); pos = np.asarray(r.scene.camera[:3], np.float32)
    assert (box[:3] <= pos - f32(R)).all() and (box[3:] >= pos + f32(R)).all()
    prims = np.ascontiguousarray(r.scene.prims); bad = {}; hits = 0; n = 0
    for acc in accs:
        rays = r.generate_rays(acc)
        assert np.unique(rays[:, :3], axis=0).shape[0] > 1   # origins spread over the lens
        t0, p0 = brute_closest(hc, prims, rays); t, p = r.trace_kernel_packet(acc)
        bad[acc] = int(differ(t, p, t0, p0).sum()); hits += int((p0 >= 0).sum()); n += len(rays)
    r.close()
    assert hits > 0.02 * n, (hits, n)
    assert not any(bad.values()), bad


@pytest.mark.gpu
@needs_gpu
def test_gpu_origin_box_holds_the_lens():
    """After SetLens the origin box holds pos -+ R, and still does after SetScene, RefitScene and a camera move."""
    sc = scenes.random_scene(3000, light_every=40)
    r = b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    R = 400.0
    def holds():
        box = r.origin_box(); pos = np.asarray(r._cam[:3], np.float32)
        return bool((box[:3] <= pos - f32(R)).all() and (box[3:] >= pos + f32(R)).all())
    assert not holds()
    r.SetLens(R, 50.0); assert holds()
    r.SetScene(scenes.random_scene(2000, light_every=40)); assert holds()
    geo = np.ascontiguousarray(r.scene.geometry).copy(); geo["position"] *= f32(0.5); r.RefitScene(geo); assert holds()
    cam = r._cam.copy(); cam[:3] += f32(3000.0); r.SetCamera(cam); assert holds()
    r.close()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("bvh", [False, True])
def test_gpu_frames_enqueued_back_to_back_equal_frames_waited_for(bvh):
    """A lens change and a focus change in mid-pipeline, samples traced ahead (one Accumulate per frame), both sides: frames enqueued back
    to back (RenderDevice, no waits) equal frames rendered by a renderer that waits after every call."""
    sc = scenes.random_scene(3000, light_every=40) if bvh else scenes.default_scene()
    flags = b2r.FLAG_FORCE_BVH if bvh else b2r.FLAG_FORCE_BRUTE
    plan = [None] * 3 + [(0.6, 40.0)] + [None] * 3 + [(0.6, 15.0)] + [None] * 3 + [(0.0, 15.0)] + [None] * 2 + [(1.2, 25.0)] + [None] * 2
    def run(wait):
        r = b2r.Renderer(sc, 128, 64, max_bounces=6, buckets=1, flags=flags)
        for step in plan:
            if step is not None: r.SetLens(*step); r.ResetAccumulator()
            r.Accumulate(1)
            if wait: r.sync(); assert r.Render()
            else: assert r.RenderDevice()
        last = r.buckets_host(); assert r.Render(); fb = r.framebuffer.copy(); r.close()
        return last, fb, None
    a_b, a_f, _ = run(False)
    b_b, b_f, _ = run(True)
    assert float(a_b.max()) > 0.0
    assert a_b.tobytes() == b_b.tobytes() and a_f.tobytes() == b_f.tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("bvh", [False, True])
def test_gpu_bucket_split_with_a_lens(bvh):
    """Contexts that split the buckets (bucket_first / bucket_stride) with a lens reproduce the single context's buckets."""
    sc = scenes.random_scene(2000, light_every=40) if bvh else scenes.default_scene()
    flags = b2r.FLAG_FORCE_BVH if bvh else b2r.FLAG_FORCE_BRUTE; K, n = 4, 8
    one = b2r.Renderer(sc, 96, 64, max_bounces=6, buckets=K, flags=flags); one.SetLens(0.5, 30.0); one.Accumulate(n); want = one.buckets_host(); one.close()
    got = np.zeros_like(want)
    for first in range(2):
        r = b2r.Renderer(sc, 96, 64, max_bounces=6, buckets=K, flags=flags, bucket_first=first, bucket_stride=2)
        r.SetLens(0.5, 30.0); r.Accumulate(n); b = r.buckets_host(); r.close()
        for k in range(K):
            if k % 2 == first: got[k] = b[k]
    assert got.tobytes() == want.tobytes()


@pytest.mark.gpu
@needs_gpu
def test_gpu_set_lens_errors():
    sc = scenes.default_scene()
    r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1); L = b2r.lib()
    for R, F in [(-1.0, 5.0), (float("nan"), 5.0), (float("inf"), 5.0), (1.0, 0.0), (1.0, -2.0), (1.0, float("nan")), (1.0, float("inf"))]:
        assert L.b2r_set_lens(r._h, R, F) == b2r.ERR_ARG, (R, F)
    assert L.b2r_set_lens(None, 1.0, 1.0) == b2r.ERR_ARG
    r.close()
    r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_REFERENCE_EXACT)
    assert L.b2r_set_lens(r._h, 0.5, 5.0) == b2r.ERR_STATE
    r.close()
