"""Smooth dielectric (B2R_FLAG_DIELECTRIC): a material with max(transmission) > 0 reflects with the Fresnel reflectance or refracts (throughput
*= transmission) with eta = 1 + IOR_minus_one, makes no light sample, and the emitter its path reaches next gets MIS weight 1 (DESIGN.md §2).
The reference carries these fields but never reads them, so there is no reference result: the routine is checked against float64 physics,
and the kernels bit for bit against the oracle's restatement. That restatement lives in tests/dielcheck/diel_oracle.cpp, which compiles the
oracle (unchanged) through the lens oracle and restates its per-tile stream loop with the ORC_DIELECTRIC branches. The product's routines run
on the CPU through tests/dielcheck/diel_taps.cpp, which compiles the host check (unchanged) with a dielectric twin of its hc_render_sample.
This module compiles both with g++ into a temporary directory.

CPU tier: the scatter routine, the host check against the oracle, white-furnace known answers, the input rule. GPU tier (-m gpu): every
kernel that shades, batching, interior-origin rays through the BVH, and the flag rules of the C ABI."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

import b2r
import oracle_py
import scenes
from conftest import have_gpu
from test_traversal_kernels import brute_closest, differ

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
needs_gpu = pytest.mark.skipif(not have_gpu(), reason="needs a CUDA device")
f32 = np.float32
ORC_DIELECTRIC = 16
ETAS = (1.0, 1.33, 1.5, 2.4)

_DIELCHECK = None
_DIELTAPS = None


def dieltaps():
    """tests/dielcheck/diel_taps.cpp (+ csrc/b2r_host.cpp) compiled once per session into a temporary directory with the host check's flags:
    the host check's hc_* taps and dc_render_sample / dc_scatter / dc_materials_valid"""
    global _DIELTAPS
    if _DIELTAPS is None:
        import tempfile
        csrc = os.path.join(ROOT, "cpu-raytracing-experiments_b200", "csrc")
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_dieltaps_"), "libdieltaps.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mavx2", "-mfma", "-fPIC", "-shared", "-I/usr/local/cuda/include", "-I", csrc,
                               os.path.join(HERE, "dielcheck", "diel_taps.cpp"), os.path.join(csrc, "b2r_host.cpp"), "-o", out])
        L = C.CDLL(out)
        vp, u32 = C.c_void_p, C.c_uint32
        L.dc_scatter.argtypes = [vp, C.c_float, C.c_float, vp]; L.dc_scatter.restype = C.c_int
        L.dc_materials_valid.argtypes = [vp, u32]; L.dc_materials_valid.restype = C.c_int
        L.hc_closest_brute.argtypes = [vp, u32, vp, u32, vp, vp]; L.hc_closest_brute.restype = None
        _DIELTAPS = L
    return _DIELTAPS


def dielcheck():
    """tests/dielcheck/diel_oracle.cpp compiled once per session into a temporary directory (the oracle's flags): orc_*, lo_*, dl_*"""
    global _DIELCHECK
    if _DIELCHECK is None:
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_dielcheck_"), "libdielcheck.so")
        subprocess.check_call(["g++", "-std=c++17", "-fPIC", "-shared", "-pthread", "-fno-fast-math", "-O2", "-mavx2", "-mfma", "-ffp-contract=off",
                               "-I", os.path.join(ROOT, "oracle"), os.path.join(HERE, "dielcheck", "diel_oracle.cpp"), "-o", out])
        L = C.CDLL(out)
        ref = oracle_py.lib()
        for name in ("orc_create", "orc_destroy", "orc_set_scene", "orc_set_camera_lookat", "orc_get_camera_raw", "orc_reset", "orc_set_accumulations",
                     "orc_read_buckets", "orc_render", "orc_read_counters", "orc_reset_counters", "orc_generate_rays"):
            fn, r = getattr(L, name), getattr(ref, name); fn.argtypes = r.argtypes; fn.restype = r.restype
        vp, f = C.c_void_p, C.c_float
        L.dl_accumulate.argtypes = [vp, C.c_uint32, C.c_int]; L.dl_accumulate.restype = None
        L.dl_scatter.argtypes = [vp, f, f, vp]; L.dl_scatter.restype = C.c_int
        L.lo_set_lens.argtypes = [vp, f, f]; L.lo_set_lens.restype = None
        _DIELCHECK = L
    return _DIELCHECK


class DielOracle(oracle_py.Oracle):
    """oracle_py.Oracle on the oracle with the dielectric restated (flags may hold ORC_DIELECTRIC); set_lens as the lens oracle's"""

    def __init__(self, width, height, max_bounces=16, K=1, flags=0):
        self.L = dielcheck()
        self.h = self.L.orc_create(width, height, max_bounces, K, flags)
        assert self.h
        self.width, self.height, self.K, self.max_bounces = width, height, K, max_bounces
        self.npix = width * height
        self.L.lo_set_lens(self.h, 0.0, 1.0)

    def accumulate(self, n=1, threads=None):
        self.L.dl_accumulate(self.h, n, threads or os.cpu_count() or 1)

    def set_lens(self, radius, focus_distance):
        self.L.lo_set_lens(self.h, radius, focus_distance)

    def sample(self, acc):
        """per-sample radiance of sample index acc (tile order) and the counters of that sample"""
        self.reset(); self.reset_counters(); self.set_accumulations(acc - 1); self.accumulate(1)
        return self.buckets()[0], self.counters()


@pytest.fixture(scope="module")
def hc():
    return dieltaps()


def render_hc(hc, sc, w, h, mb, acc, use_bvh, flags=0):
    """one sample of every pixel through dc_render_sample (the kernels' shading routines on the host): (rad[3][npix] tile order, counters)"""
    ps = b2r.PreparedScene(sc, w, h)
    rad = np.zeros((3, w * h), np.float32); cnt = (C.c_uint64 * 5)()
    vp = lambda a: C.c_void_p(a.ctypes.data)
    rc = hc.dc_render_sample(vp(ps.prims), vp(ps.nodes), len(ps.prims), len(ps.nodes), vp(ps.material), len(ps.material), vp(ps.lights), len(ps.lights),
                             vp(ps.geometry), vp(ps.camera), w, h, mb, flags, acc, use_bvh, vp(rad), cnt,
                             vp(ps.ambient), None if ps.hdri is None else vp(ps.hdri), 0 if ps.hdri is None else ps.hdri.shape[1], 0 if ps.hdri is None else ps.hdri.shape[0])
    assert rc == 0
    return rad, list(cnt)


def _p(a):
    return C.c_void_p(a.ctypes.data)


def _glass(sc, mats, eta=1.5, t=(0.95, 0.95, 0.95)):
    """sc with the materials `mats` turned to glass (a copy)"""
    sc = scenes.Scene(sc); m = np.ascontiguousarray(sc["material"]).copy()
    for k in mats:
        m[k]["transmission"] = np.asarray(t, f32); m[k]["IOR_minus_one"] = f32(eta - 1.0)
    sc["material"] = m
    return sc


def _furnace(t, eta):
    return _glass(scenes.white_furnace(), [0], eta, t)


def _nested(inner_emits):
    """a glass sphere (IOR 1.5) holding a smaller diffuse sphere or a smaller emitter, lit by a light outside"""
    mats = [scenes._mat(albedo=[0.1, 0.1, 0.1], transmission=[0.9, 0.95, 1.0], IOR_minus_one=f32(0.5)),
            scenes._mat(albedo=[0.8, 0.3, 0.2], emission=[6.0, 5.0, 4.0] if inner_emits else [0, 0, 0]),
            scenes._mat(emission=[20.0, 20.0, 20.0]), scenes._mat(albedo=[0.6, 0.6, 0.6])]
    geo = [scenes._sphere((0, 0, 0), 1.0, 0), scenes._sphere((0.1, -0.1, 0.0), 0.16, 1), scenes._sphere((2.5, 3.0, 1.0), 0.25, 2),
           scenes._sphere((0, -1001.2, 0), 1e6, 3)]
    return scenes.Scene(name="nested", geometry=np.array(geo, dtype=scenes.SPHERE_DTYPE), material=np.array(mats, dtype=scenes.MATERIAL_DTYPE),
                        camera=dict(eye=(0.3, 0.4, 3.2), dir=(-0.1, -0.12, -1), focal_length=40.0, exposure=1.0), ambient=(0.0, 0.0, 0.0))


def _tir_scene():
    """eta = 2.4 spheres seen at grazing incidence along a floor: most paths inside them are totally reflected"""
    sc = _glass(scenes.default_scene(), [], 2.4)
    m = np.ascontiguousarray(sc["material"]).copy(); g = np.ascontiguousarray(sc["geometry"])
    lit = set(int(k) for k in g["material_ID"] if m[k]["emission"].max() > 0)
    for k in range(len(m)):
        if k not in lit and k != int(g["material_ID"][np.argmax(g["radius_sq"])]):   # everything but the lights and the ground
            m[k]["transmission"] = np.asarray([1.0, 0.9, 0.8], f32); m[k]["IOR_minus_one"] = f32(1.4)
    sc["material"] = m
    eye = np.asarray(sc["camera"]["eye"], np.float64); eye[1] = float(g["position"][:, 1][np.argmax(g["radius_sq"])] + np.sqrt(g["radius_sq"].max())) + 0.05
    sc["camera"] = dict(sc["camera"], eye=tuple(eye), dir=(float(-eye[0]), -0.02, float(-eye[2])))
    return sc


def _glass_random(n=1500, ggx=False):
    """a random scene with two of its materials made glass (IOR 1.5, transmission 0.95)"""
    sc = scenes.ggx_random_scene(n) if ggx else scenes.random_scene(n, light_every=40)
    return _glass(sc, [1, 4])


CPU_SCENES = {"default": scenes.default_scene, "random": _glass_random, "nested_diffuse": lambda: _nested(False), "nested_emitter": lambda: _nested(True),
              "tir": _tir_scene}


def _rand_v(rs, n):
    v = rs.randn(n, 3); v[:, 2] = np.abs(v[:, 2]); v /= np.linalg.norm(v, axis=1, keepdims=True)
    v[:4] = [[0, 0, 1], [1e-4, 0, 1], [0.6, 0.8, 1e-7], [0.8, 0, 0.6]]
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(f32)


def _scatter(hc, v, r, u0):
    out = np.zeros(4, f32); vv = np.ascontiguousarray(v, f32)
    refl = hc.dc_scatter(_p(vv), f32(r), f32(u0), _p(out))
    return bool(refl), out[:3].copy(), float(out[3])


def _fresnel_conditioning(c, r):
    """bound of F's float error from the rounding of ct = sqrt(1 - s2): |d ct| <= ~2u / ct, and |dF| <= 2 |d Rs| + 2 |d Rp| with |dR / d ct| <=
    2 / (the sum in its denominator); large only near grazing incidence and near the critical angle"""
    s2 = r * r * (1 - c * c)
    if s2 >= 1: return 0.0
    ct = np.sqrt(1 - s2); u = 2.0 ** -24
    return 8 * (2 * u / ct) / min(r * c + ct, r * ct + c)


def _fresnel64(c, r):
    s2 = r * r * (1 - c * c)
    if s2 >= 1: return 1.0
    ct = np.sqrt(1 - s2); rs = (r * c - ct) / (r * c + ct); rp = (r * ct - c) / (r * ct + c)
    return 0.5 * (rs * rs + rp * rp)


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("eta", ETAS)
def test_scatter_routine_against_float64_physics(hc, eta):
    """dielectric_scatter (the kernels' routine, on the host) on random unit v_local, entering (r = 1/eta) and leaving (r = eta): the reflection
    is the mirror direction, the refraction obeys Snell's law (r sin(theta_i) = sin(theta_t) to a few ulps), F is the float64 Fresnel formula,
    total internal reflection gives F = 1 and reflects at u0 = 1.0; the oracle's restatement returns the same bits (grazing v_local too, where
    the float64 comparisons are skipped: below v.z ~ 2.4e-4, 1 - v.z^2 rounds to 1)."""
    rs = np.random.RandomState(int(eta * 100)); V = _rand_v(rs, 400); dl = dielcheck()
    for leaving in (False, True):
        r = f32(eta) if leaving else f32(1.0) / f32(eta)
        for v in V:
            c = float(min(max(v[2], 0.0), 1.0)); F64 = _fresnel64(np.float64(c), np.float64(r))
            for u0 in (0.0, float(rs.rand()), 1.0):
                refl, d, F = _scatter(hc, v, r, u0)
                o = np.zeros(4, f32); assert bool(dl.dl_scatter(_p(np.ascontiguousarray(v)), r, f32(u0), _p(o))) == refl
                assert o.tobytes() == np.r_[d, f32(F)].astype(f32).tobytes()
                if c < 1e-3:   # grazing: 1 - c^2 rounds to 1 in float (c < ~2.4e-4), so r >= 1 reads as total internal reflection (DESIGN §2)
                    continue
                assert abs(F - F64) <= 2e-6 + 1e-5 * F64 + _fresnel_conditioning(c, float(r)), (v, r, F, F64)
                if F64 == 1.0:
                    assert F == 1.0 and refl
                assert refl == (F64 == 1.0 or u0 < F)
                if refl:
                    assert d.tobytes() == np.array([-v[0], -v[1], c], f32).tobytes()
                else:
                    d64 = d.astype(np.float64)
                    sin_t = np.hypot(d64[0], d64[1]) / np.linalg.norm(d64); sin_i = np.hypot(float(v[0]), float(v[1]))
                    assert abs(float(r) * sin_i - sin_t) <= 8 * 2.0 ** -24, (v, r)
                    assert d[2] < 0 and abs(np.linalg.norm(d64) - 1.0) <= 8 * 2.0 ** -24
    # normal incidence: ((eta - 1) / (eta + 1))^2 both ways
    for r in (f32(eta), f32(1.0) / f32(eta)):
        _, _, F = _scatter(hc, [0, 0, 1], r, 0.5)
        assert abs(F - ((eta - 1) / (eta + 1)) ** 2) <= 1e-6
    if eta == 1.0:   # index matched: no reflection, the ray goes straight on
        for v in V[V[:, 2] >= 1e-3]:
            refl, d, F = _scatter(hc, v, 1.0, 0.5)
            c = float(v[2]); assert not refl and F <= 2e-6 + _fresnel_conditioning(c, 1.0)
            assert np.abs(d[:2] + v[:2]).max() == 0.0 and abs(float(d[2]) + c) <= 4 * 2.0 ** -24 + 2 * 2.0 ** -24 / c   # ct = sqrt(1 - (1 - c^2)): rounding / c
    else:            # leaving beyond the critical angle: total internal reflection whatever u0 is
        c = 0.5 * np.sqrt(1 - 1 / eta ** 2); v = np.array([np.sqrt(1 - c * c), 0, c], f32)
        refl, d, F = _scatter(hc, v, eta, 1.0)
        assert refl and F == 1.0


@pytest.mark.parametrize("name", list(CPU_SCENES))
@pytest.mark.parametrize("ggx", [False, True])
def test_host_check_equals_the_oracle_bit_for_bit(hc, name, ggx):
    """dc_render_sample with the flag (the kernels' shading routines on the host) == the oracle's ORC_DIELECTRIC frames bit for bit, with and
    without GGX, brute force and the traversal tree; the default scene, a random scene with glass, a glass sphere holding a diffuse sphere or
    an emitter, and a TIR-heavy scene (eta = 2.4, grazing camera). The paths really meet glass: the glass frames differ from opaque ones."""
    sc = CPU_SCENES[name](); w, h, mb = 128, 80, 12
    flags = b2r.FLAG_DIELECTRIC | (b2r.FLAG_GGX if ggx else 0)
    o = DielOracle(w, h, max_bounces=mb, flags=ORC_DIELECTRIC | (oracle_py.ORC_GGX if ggx else 0)); o.set_scene(sc)
    for acc, use_bvh in ((1, 0), (9, 2)):
        ref, oc = o.sample(acc)
        rad, cnt = render_hc(hc, sc, w, h, mb, acc, use_bvh, flags)
        assert rad.tobytes() == ref.tobytes(), (acc, use_bvh)
        assert cnt[0] == oc["extension_rays"] and cnt[2] == oc["shaded_hits"] and cnt[3] == oc["terminated"] and cnt[4] == oc["dropped"]
        opaque, _ = render_hc(hc, sc, w, h, mb, acc, use_bvh, flags & ~b2r.FLAG_DIELECTRIC)
        assert opaque.tobytes() != rad.tobytes()
    o.close()


def test_oracle_restatement_without_the_flag_is_the_oracle(hc):
    """The restated stream loop without ORC_DIELECTRIC == the oracle's own loop, bit for bit (default scene with its glass materials, GGX too)."""
    sc = scenes.default_scene(); w, h, mb = 96, 64, 8
    for of in (0, oracle_py.ORC_GGX):
        a = DielOracle(w, h, max_bounces=mb, K=2, flags=of); a.set_scene(sc); a.accumulate(3)
        b = oracle_py.Oracle(w, h, max_bounces=mb, K=2, flags=of); b.set_scene(sc); b.accumulate(3)
        assert a.buckets().tobytes() == b.buckets().tobytes()
        a.close(); b.close()


def _furnace_check(rad, dropped):
    px = rad.T   # [npix][3]
    assert np.isin(px, (0.0, 1.0)).all()
    zeros = np.all(px == 0.0, axis=1)
    assert (np.all(px == 1.0, axis=1) | zeros).all()
    assert int(zeros.sum()) == dropped
    return int(zeros.sum())


def test_white_furnace_with_glass(hc):
    """White furnace, its sphere made clear glass (transmission 1, IOR 1.5): every per-sample linear pixel is exactly the ambient 1.0, except
    paths dropped at max_bounces (Q11), which are exactly 0, as many as the dropped-path counter says; oracle and host check."""
    sc = _furnace((1.0, 1.0, 1.0), 1.5); w, h, mb = 64, 64, 3; flags = b2r.FLAG_DIELECTRIC   # mb = 3: one internal reflection drops a path
    o = DielOracle(w, h, max_bounces=mb, flags=ORC_DIELECTRIC); o.set_scene(sc)
    dropped = 0
    for acc in (1, 2, 3):
        ref, oc = o.sample(acc)
        dropped += _furnace_check(ref, oc["dropped"])
        for use_bvh in (0, 2):
            rad, cnt = render_hc(hc, sc, w, h, mb, acc, use_bvh, flags)
            assert rad.tobytes() == ref.tobytes()
            _furnace_check(rad, cnt[4])
    assert dropped > 0
    o.close()


def _sphere_masks(o, acc, margin=0.02):
    """pixels whose camera ray (sample acc) passes the unit sphere at the origin well inside / well outside its silhouette (float64)"""
    rays = o.generate_rays(acc).astype(np.float64); orig, d = rays[:, :3], rays[:, 3:]
    d = d / np.linalg.norm(d, axis=1, keepdims=True)
    t = -np.einsum("ij,ij->i", orig, d); p = np.linalg.norm(orig + t[:, None] * d, axis=1)
    return p < 1.0 - margin, p > 1.0 + margin


def test_index_matched_sphere(hc):
    """eta = 1, transmission 0.9 in the white furnace: a camera ray through the sphere refracts twice without bending, so the converged mean
    inside the silhouette is 0.81 (each sample is 0 or about 1 after roulette's compensation; the bound is 5 standard deviations of that
    mean); pixels outside the silhouette are exactly 1."""
    sc = _furnace((0.9, 0.9, 0.9), 1.0); w, h, mb = 64, 64, 8
    o = DielOracle(w, h, max_bounces=mb, flags=ORC_DIELECTRIC); o.set_scene(sc)
    vals = []
    for acc in range(1, 33):
        ref, _ = o.sample(acc)
        inside, outside = _sphere_masks(o, acc)
        assert (ref[:, outside] == 1.0).all()
        vals.append(ref[0, inside].astype(np.float64))
        if acc <= 2:
            rad, _ = render_hc(hc, sc, w, h, mb, acc, 0, b2r.FLAG_DIELECTRIC); assert rad.tobytes() == ref.tobytes()
    v = np.concatenate(vals); bound = 5.0 * np.sqrt(0.81 * 0.19 / len(v))
    assert abs(v.mean() - 0.81) <= bound, (v.mean(), bound, len(v))
    o.close()


def _bad_materials():
    """(name, material array) pairs that break the dielectric input rule"""
    base = scenes.default_scene()["material"]
    out = []
    for name, t, iorm1 in [("nan_t", (np.nan, 0.5, 0.5), 0.5), ("inf_t", (0.2, np.inf, 0.2), 0.5), ("t_above_1", (1.5, 0.5, 0.5), 0.5),
                           ("t_below_0", (-0.1, 0.5, 0.5), 0.5), ("eta_below_1", (0.5, 0.5, 0.5), -0.5), ("eta_nan", (0.5, 0.5, 0.5), np.nan),
                           ("eta_inf", (0.5, 0.5, 0.5), np.inf), ("nan_t_not_glass", (np.nan, 0.0, 0.0), 0.0)]:
        m = np.ascontiguousarray(base).copy(); m[2]["transmission"] = np.asarray(t, f32); m[2]["IOR_minus_one"] = f32(iorm1); out.append((name, m))
    return out


def test_input_rule_on_the_host(hc):
    """dielectric_materials_valid, the rule b2r_upload_scene / b2r_refit_scene / b2r_set_flags apply under the flag: the scenes' materials
    pass, each bad material fails, and so do eta exactly 1 and transmission exactly 0 or 1 pass."""
    for sc in (scenes.default_scene(), _furnace((1, 1, 1), 1.0), _tir_scene(), scenes.random_scene(100)):
        m = np.ascontiguousarray(sc["material"]); assert hc.dc_materials_valid(_p(m), len(m)) == 1
    for name, m in _bad_materials():
        assert hc.dc_materials_valid(_p(m), len(m)) == 0, name


def test_flag_with_reference_exact_is_refused_at_create():
    """B2R_FLAG_DIELECTRIC | B2R_FLAG_REFERENCE_EXACT is B2R_ERR_ARG at b2r_create, before any device is needed."""
    cfg = b2r.Config(64, 48, 4, 1, b2r.FLAG_DIELECTRIC | b2r.FLAG_REFERENCE_EXACT, 0, 0, 0, 0)
    h = C.c_void_p(None)
    assert b2r.lib().b2r_create(C.byref(h), C.byref(cfg)) == b2r.ERR_ARG
    assert not h.value


# ------------------------------------------------------------------------------------------------ GPU tier
def _gpu_vs_oracle(sc, w, h, mb, flags, lens=None, n=2):
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags | b2r.FLAG_DIELECTRIC)
    o = DielOracle(w, h, max_bounces=mb, flags=ORC_DIELECTRIC | (oracle_py.ORC_GGX if flags & b2r.FLAG_GGX else 0)); o.set_scene(sc)
    if lens: r.SetLens(*lens); o.set_lens(*lens)
    r.Accumulate(n); o.accumulate(n)
    got, want = r.buckets_host(), o.buckets(); r.close(); o.close()
    assert float(want.max()) > 0.0
    return got, want


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("case", ["default_brute", "default_bvh", "glass1500_bvh", "default_lens_brute", "default_lens_bvh"])
@pytest.mark.parametrize("ggx", [False, True])
def test_gpu_equals_the_oracle(case, ggx):
    """Every kernel that shades (k_bounce_brute with its FIRST and LENS variants, k_brute_finish, k_shade) with the flag, bit for bit against
    the oracle's ORC_DIELECTRIC frames: the default scene at 128x80 in both pipelines, a 1500-sphere glass scene in the BVH pipeline, the
    default scene with a lens; with and without GGX."""
    g = b2r.FLAG_GGX if ggx else 0
    if case.startswith("glass1500"):
        got, want = _gpu_vs_oracle(_glass_random(1500, ggx), 160, 96, 8, g | b2r.FLAG_FORCE_BVH)
    else:
        pipe = b2r.FLAG_FORCE_BRUTE if case.endswith("brute") else b2r.FLAG_FORCE_BVH
        got, want = _gpu_vs_oracle(scenes.default_scene(), 128, 80, 12, g | pipe, lens=(0.3, 4.5) if "lens" in case else None)
    assert got.tobytes() == want.tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("bvh", [False, True])
@pytest.mark.parametrize("ggx", [False, True])
def test_gpu_scene_without_glass_is_unchanged(bvh, ggx):
    """On a scene with no transmissive material, frames with the flag are bit-identical to frames without it."""
    sc = scenes.Scene(scenes.default_scene()); m = np.ascontiguousarray(sc["material"]).copy(); m["transmission"] = 0.0; sc["material"] = m
    flags = (b2r.FLAG_FORCE_BVH if bvh else b2r.FLAG_FORCE_BRUTE) | (b2r.FLAG_GGX if ggx else 0)
    out = []
    for f in (flags, flags | b2r.FLAG_DIELECTRIC):
        r = b2r.Renderer(sc, 128, 80, max_bounces=10, buckets=2, flags=f); r.Accumulate(4); out.append(r.buckets_host()); r.close()
    assert float(out[0].max()) > 0.0 and out[0].tobytes() == out[1].tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("bvh", [False, True])
def test_gpu_batching_changes_no_bits(bvh):
    """Full-width batches == one sample in flight without the graph; frames enqueued back to back == frames waited for; b2r_refit_scene after
    moving the glass spheres == a fresh upload of the moved scene."""
    sc = _glass_random(1500) if bvh else scenes.default_scene()
    flags = (b2r.FLAG_FORCE_BVH if bvh else b2r.FLAG_FORCE_BRUTE) | b2r.FLAG_DIELECTRIC; w, h, mb = 128, 80, 10
    def run(**kw):
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=2, **kw); r.Accumulate(6); b = r.buckets_host(); r.close(); return b
    want = run(flags=flags)
    assert float(want.max()) > 0.0
    assert run(flags=flags | b2r.FLAG_NO_GRAPH, samples_in_flight=1).tobytes() == want.tobytes()
    def frames(wait):
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags)
        for _ in range(8):
            r.Accumulate(1)
            if wait: r.sync(); assert r.Render()
            else: assert r.RenderDevice()
        b = r.buckets_host(); assert r.Render(); fb = r.framebuffer.copy(); r.close(); return b, fb
    a, b = frames(False), frames(True)
    assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()
    geo = np.ascontiguousarray(sc["geometry"]).copy(); m = np.ascontiguousarray(sc["material"])
    glass = m["transmission"][geo["material_ID"]].max(axis=1) > 0
    assert glass.any()
    geo["position"][glass] += np.asarray([0.3, 0.2, -0.1], f32)
    moved = scenes.Scene(sc); moved["geometry"] = geo
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags); r.Accumulate(2); r.RefitScene(geo); r.ResetAccumulator(); r.Accumulate(3)
    got = r.buckets_host(); r.close()
    r = b2r.Renderer(moved, w, h, max_bounces=mb, buckets=1, flags=flags); r.Accumulate(3); fresh = r.buckets_host(); r.close()
    assert got.tobytes() == fresh.tobytes()


def _interior_rays(sc, seed=31):
    """for every sphere: a point on its surface (random normal N), one ray from hit - 1e-4 N going inward and one from hit + 1e-4 N going outward"""
    g = np.ascontiguousarray(sc["geometry"]); rs = np.random.RandomState(seed); n = len(g)
    N = rs.randn(n, 3); N /= np.linalg.norm(N, axis=1, keepdims=True)
    c = g["position"].astype(np.float64); r = np.sqrt(g["radius_sq"].astype(np.float64))[:, None]
    hit = c + r * N
    def dirs(sign):
        d = rs.randn(n, 3); d /= np.linalg.norm(d, axis=1, keepdims=True)
        dn = np.einsum("ij,ij->i", d, N)[:, None]; return np.where(sign * dn >= 0, d, d - 2 * dn * N)
    rin = np.concatenate([(hit - 1e-4 * N), dirs(-1.0)], axis=1); rout = np.concatenate([(hit + 1e-4 * N), dirs(1.0)], axis=1)
    return np.ascontiguousarray(np.concatenate([rin, rout]), f32)


def _brute_closest_parallel(hc, prims, rays):
    """hc_closest_brute over chunks of the rays on every core (ctypes releases the GIL during the call)"""
    t = np.empty(len(rays), f32); p = np.empty(len(rays), np.int32); k = os.cpu_count() or 1; edges = np.linspace(0, len(rays), k + 1).astype(int)
    def work(a, b):
        tt, pp = brute_closest(hc, prims, np.ascontiguousarray(rays[a:b])); t[a:b] = tt; p[a:b] = pp
    th = [threading.Thread(target=work, args=(edges[i], edges[i + 1])) for i in range(k) if edges[i] < edges[i + 1]]
    for x in th: x.start()
    for x in th: x.join()
    return t, p


@pytest.mark.gpu
@needs_gpu
def test_gpu_bvh_equals_brute_force_on_interior_origin_rays(hc):
    """Refraction starts rays 1e-4 inside a sphere, which no earlier shading event did routinely. On C3's scene, rays from hit - 1e-4 N going
    inward and from hit + 1e-4 N going outward, for every sphere, through k_intersect_closest (b2r_trace_kernel) == brute force: zero
    divergent rays."""
    sc = scenes.random_scene(100000); rays = _interior_rays(sc)
    r = b2r.Renderer(sc, 128, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | b2r.FLAG_DIELECTRIC)
    t, p = r.trace_kernel_closest(rays); prims = np.ascontiguousarray(r.scene.prims); r.close()
    t0, p0 = _brute_closest_parallel(hc, prims, rays)
    assert (p0 >= 0).mean() > 0.9
    assert int(differ(t, p, t0, p0).sum()) == 0


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("bvh", [False, True])
def test_gpu_white_furnace_with_glass(bvh):
    """The two furnace known answers on the GPU: clear glass gives exactly 1 or (dropped) exactly 0, zeros == the dropped counter; the
    index-matched sphere converges to 0.81 inside its silhouette and is exactly 1 outside."""
    flags = (b2r.FLAG_FORCE_BVH if bvh else b2r.FLAG_FORCE_BRUTE) | b2r.FLAG_DIELECTRIC | b2r.FLAG_NO_SPECULATION; w = h = 64
    sc = _furnace((1.0, 1.0, 1.0), 1.5); dropped = 0
    r = b2r.Renderer(sc, w, h, max_bounces=3, buckets=1, flags=flags)
    for _ in range(3):   # per sample: the bucket sums are small integers, so their differences are exact
        before, d0 = r.buckets_host()[0].copy(), r.counters()["dropped"]; r.Accumulate(1)
        dropped += _furnace_check(r.buckets_host()[0] - before, r.counters()["dropped"] - d0)
    r.close()
    assert dropped > 0
    sc = _furnace((0.9, 0.9, 0.9), 1.0); o = DielOracle(w, h, max_bounces=8, flags=ORC_DIELECTRIC); o.set_scene(sc)
    r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=1, flags=flags); vals = []
    for acc in range(1, 33):
        before = r.buckets_host()[0].copy(); r.Accumulate(1); rad = r.buckets_host()[0] - before
        inside, outside = _sphere_masks(o, acc)
        assert (rad[:, outside] == 1.0).all()
        vals.append(rad[0, inside].astype(np.float64))
    r.close(); o.close()
    v = np.concatenate(vals); bound = 5.0 * np.sqrt(0.81 * 0.19 / len(v))
    assert abs(v.mean() - 0.81) <= bound, (v.mean(), bound)


@pytest.mark.gpu
@needs_gpu
def test_gpu_flag_rules(tmp_path):
    """The C ABI's rules: REFERENCE_EXACT with the flag at b2r_create and at b2r_set_flags; each bad material at upload and at refit with the
    flag, and at b2r_set_flags turning the flag on (the flags then stay as they were); the same materials without the flag as today; no
    checkpoint across the flag."""
    sc = scenes.default_scene(); L = b2r.lib()
    with pytest.raises(b2r.B2RError) as e:
        b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_DIELECTRIC | b2r.FLAG_REFERENCE_EXACT)
    assert e.value.code == b2r.ERR_ARG
    r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_REFERENCE_EXACT)
    assert L.b2r_set_flags(r._h, b2r.FLAG_REFERENCE_EXACT | b2r.FLAG_DIELECTRIC) == b2r.ERR_ARG
    r.close()
    for name, m in _bad_materials():
        bad = scenes.Scene(sc); bad["material"] = m
        with pytest.raises(b2r.B2RError) as e:
            b2r.Renderer(bad, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_DIELECTRIC)
        assert e.value.code == b2r.ERR_ARG, name
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_DIELECTRIC)
        with pytest.raises(b2r.B2RError) as e:
            r.RefitScene(sc["geometry"], material=m)
        assert e.value.code == b2r.ERR_ARG, name
        r.close()
        r = b2r.Renderer(bad, 64, 48, max_bounces=4, buckets=1)   # accepted without the flag, refit too
        r.RefitScene(sc["geometry"], material=m); r.Accumulate(1)
        assert L.b2r_set_flags(r._h, b2r.FLAG_DIELECTRIC) == b2r.ERR_ARG, name
        r.close()
    # a refused set_flags leaves the flags as they were: the frame equals one of a context that never had the flag
    bad = scenes.Scene(sc); bad["material"] = _bad_materials()[2][1]
    r = b2r.Renderer(bad, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BRUTE)
    assert L.b2r_set_flags(r._h, b2r.FLAG_FORCE_BRUTE | b2r.FLAG_DIELECTRIC) == b2r.ERR_ARG
    r.Accumulate(2); got = r.buckets_host(); r.close()
    r = b2r.Renderer(bad, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BRUTE); r.Accumulate(2); want = r.buckets_host(); r.close()
    assert got.tobytes() == want.tobytes()
    # checkpoints do not cross the flag, either way
    for a, b in ((b2r.FLAG_DIELECTRIC, 0), (0, b2r.FLAG_DIELECTRIC)):
        path = tmp_path / f"ck_{a}_{b}.b2r"
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=a); r.Accumulate(2); r.SaveCheckpoint(path); r.close()
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b)
        assert L.b2r_load_checkpoint(r._h, str(path).encode()) == b2r.ERR_STATE
        r.close()
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=a); r.LoadCheckpoint(path); r.close()   # same flags: loads
