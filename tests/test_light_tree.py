"""Sphere lights picked by importance from a light tree (B2R_FLAG_LIGHT_TREE): next-event estimation descends a binary tree over the light list
instead of picking uniformly, and both MIS weights use the tree's pdf (DESIGN.md §2). The reference picks uniformly, so there is no reference
result: the builder and the pdf are checked against their definition, and the kernels bit for bit against the oracle's restatement. That
restatement lives in tests/ltreecheck/ltree_oracle.cpp, which compiles the oracle (unchanged) through the sky, dielectric and lens
restatements and adds the ORC_LIGHT_TREE branches; the product's routines and the host builder run on the CPU through
tests/ltreecheck/ltree_taps.cpp. This module compiles both with g++ into a temporary directory.

CPU tier: builder, selection pdf and descent, MIS complement, host check against the restatement, known answers, unbiasedness, payoff, the
create-time refusals. GPU tier (-m gpu): every kernel that shades, batching, context operations, full-size unbiasedness, the C ABI's rules."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import b2r
import oracle_py
import scenes
from conftest import have_gpu
from test_sky_light import SkyOracle, render_taps as sky_render_taps, _sun, _default_sky, ORC_DIELECTRIC, ORC_SKY_LIGHT

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
needs_gpu = pytest.mark.skipif(not have_gpu(), reason="needs a CUDA device")
f32 = np.float32
ORC_NO_MIS, ORC_GGX, ORC_LIGHT_TREE = 4, 8, 64

_TAPS = None
_ORACLE = None


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def taps():
    """tests/ltreecheck/ltree_taps.cpp (+ csrc/b2r_host.cpp) with the host check's flags, compiled once per session into a temporary directory"""
    global _TAPS
    if _TAPS is None:
        import tempfile
        csrc = os.path.join(ROOT, "cpu-raytracing-experiments_b200", "csrc")
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_ltreetaps_"), "libltreetaps.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mavx2", "-mfma", "-fPIC", "-shared", "-I/usr/local/cuda/include", "-I", csrc,
                               os.path.join(HERE, "ltreecheck", "ltree_taps.cpp"), os.path.join(csrc, "b2r_host.cpp"), "-o", out])
        L = C.CDLL(out)
        vp, u32 = C.c_void_p, C.c_uint32
        L.lt_list_valid.argtypes = [vp, vp, u32, vp]; L.lt_list_valid.restype = C.c_int
        L.lt_build.argtypes = [vp, vp, u32, vp, u32, vp, vp, vp, vp, vp, vp]; L.lt_build.restype = u32
        L.lt_pick.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp]; L.lt_pick.restype = None
        L.lt_pdf_all.argtypes = [vp, vp, u32, vp, vp]; L.lt_pdf_all.restype = None
        L.lt_sel_pair.argtypes = [vp, vp, vp, C.c_float, vp, vp, u32, vp, vp, vp]; L.lt_sel_pair.restype = None
        _TAPS = L
    return _TAPS


def oracle_lib():
    """tests/ltreecheck/ltree_oracle.cpp compiled once per session into a temporary directory (the oracle's flags)"""
    global _ORACLE
    if _ORACLE is None:
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_ltreecheck_"), "libltreecheck.so")
        subprocess.check_call(["g++", "-std=c++17", "-fPIC", "-shared", "-pthread", "-fno-fast-math", "-O2", "-mavx2", "-mfma", "-ffp-contract=off",
                               "-I", os.path.join(ROOT, "oracle"), os.path.join(HERE, "ltreecheck", "ltree_oracle.cpp"), "-o", out])
        L = C.CDLL(out)
        ref = oracle_py.lib()
        for name in ("orc_create", "orc_destroy", "orc_set_scene", "orc_set_camera_lookat", "orc_get_camera_raw", "orc_reset", "orc_set_accumulations",
                     "orc_read_buckets", "orc_render", "orc_read_counters", "orc_reset_counters", "orc_generate_rays"):
            fn, r = getattr(L, name), getattr(ref, name); fn.argtypes = r.argtypes; fn.restype = r.restype
        vp, f = C.c_void_p, C.c_float
        L.sk_accumulate.argtypes = [vp, C.c_uint32, C.c_int]; L.sk_accumulate.restype = None
        L.lt_accumulate.argtypes = [vp, C.c_uint32, C.c_int]; L.lt_accumulate.restype = None
        L.sk_set_tables.argtypes = [vp, vp, vp, vp, C.c_uint32, C.c_uint32]; L.sk_set_tables.restype = None
        L.lt_set_tree.argtypes = [vp, vp, C.c_uint32]; L.lt_set_tree.restype = None
        L.lo_set_lens.argtypes = [vp, f, f]; L.lo_set_lens.restype = None
        _ORACLE = L
    return _ORACLE


def light_arrays(ps):
    """the light list as the builder takes it: geometry[lights] and the mean emission of each light's material"""
    ls = np.ascontiguousarray(ps.geometry[ps.lights])
    lum = ((ps.material["emission"][ls["material_ID"]].astype(f32).sum(axis=1, dtype=f32)) / f32(3.0)).astype(f32)
    return ls, np.ascontiguousarray(lum)


def build(lights, lum, prims):
    """the host builder: (nodes[N][8], light[n][4], prim_light[n_prims], lo[N][3], hi[N][3], depth)"""
    L = taps(); n, n_prims = len(lights), len(prims)
    lights = np.ascontiguousarray(lights, scenes.SPHERE_DTYPE); prims = np.ascontiguousarray(prims, scenes.SPHERE_DTYPE); lum = np.ascontiguousarray(lum, f32)
    N = L.lt_build(_p(lights), _p(lum), n, _p(prims), n_prims, None, None, None, None, None, None)
    nodes = np.zeros((N, 8), f32); light = np.zeros((n, 4), np.int32); pl = np.zeros(n_prims, np.int32)
    lo = np.zeros((N, 3), f32); hi = np.zeros((N, 3), f32); depth = C.c_uint32(0)
    L.lt_build(_p(lights), _p(lum), n, _p(prims), n_prims, _p(nodes), _p(light), _p(pl), _p(lo), _p(hi), C.byref(depth))
    return nodes, light, pl, lo, hi, depth.value


def build_ps(ps):
    ls, lum = light_arrays(ps)
    return build(ls, lum, ps.prims)


def links(nodes):
    return np.ascontiguousarray(nodes[:, 5]).view(np.int32)


def pdf_all(nodes, light, P):
    out = np.zeros(len(light), f32); taps().lt_pdf_all(_p(nodes), _p(light), len(light), _p(np.asarray(P, f32)), _p(out)); return out


def pick(nodes, light, P, u):
    P = np.ascontiguousarray(P, f32); u = np.ascontiguousarray(u, f32); m = len(u)
    k = np.zeros(m, np.int32); pdf = np.zeros(m, f32); pdf_of = np.zeros(m, f32)
    taps().lt_pick(_p(nodes), _p(light), _p(P), _p(u), m, _p(k), _p(pdf), _p(pdf_of))
    return k, pdf, pdf_of


def _random_lights(n, seed, coincident=False, zero=False):
    rs = np.random.RandomState(seed)
    g = np.zeros(n, scenes.SPHERE_DTYPE)
    g["position"] = (rs.rand(n, 3) * [200, 100, 200]).astype(f32) if not coincident else f32([1.0, 2.0, 3.0])
    g["radius_sq"] = (rs.rand(n) * 4 + 0.01).astype(f32) ** 2
    g["material_ID"] = np.arange(n) % 3
    lum = np.zeros(n, f32) if zero else (rs.rand(n) * 20).astype(f32)
    return g, lum


class LtOracle(SkyOracle):
    """SkyOracle on the oracle with the light tree restated (flags may hold ORC_LIGHT_TREE); the host builder's tree"""

    def __init__(self, width, height, max_bounces=16, K=1, flags=0):
        self.L = oracle_lib()
        self.h = self.L.orc_create(width, height, max_bounces, K, flags)
        assert self.h
        self.width, self.height, self.K, self.max_bounces, self.flags = width, height, K, max_bounces, flags
        self.npix = width * height
        self.L.lo_set_lens(self.h, 0.0, 1.0)

    def set_scene(self, sc):
        n = super().set_scene(sc)
        ps = b2r.PreparedScene(sc, self.width, self.height)
        if (self.flags & ORC_LIGHT_TREE) and len(ps.lights):
            self._nodes = build_ps(ps)[0]
            self.L.lt_set_tree(self.h, _p(self._nodes), len(self._nodes))
        else:
            self.L.lt_set_tree(self.h, None, 0)
        return n

    def close(self):
        self.L.lt_set_tree(self.h, None, 0)
        super().close()

    def accumulate(self, n=1, threads=None):
        self.L.lt_accumulate(self.h, n, threads or os.cpu_count() or 1)


def render_taps(sc, w, h, mb, acc, use_bvh, flags, lens=None):
    """one sample of every pixel through lt_render_sample (the kernels' LTREE shading routines on the host): rad[3][npix] in tile order"""
    ps = b2r.PreparedScene(sc, w, h)
    rad = np.zeros((3, w * h), f32); cnt = (C.c_uint64 * 5)()
    ln = None if lens is None else np.asarray(lens, f32)
    rc = taps().lt_render_sample(_p(ps.prims), _p(ps.nodes), len(ps.prims), len(ps.nodes), _p(ps.material), len(ps.material), _p(ps.lights), len(ps.lights),
                                 _p(ps.geometry), _p(ps.camera), w, h, mb, flags, acc, use_bvh, _p(rad), cnt,
                                 _p(ps.ambient), _p(ps.hdri), 0 if ps.hdri is None else ps.hdri.shape[1], 0 if ps.hdri is None else ps.hdri.shape[0], _p(ln))
    assert rc == 0
    return rad


def _gray(sc, keep_emission=True):
    sc = scenes.Scene(sc); m = np.ascontiguousarray(sc["material"]).copy()
    m["albedo"] = m["albedo"].mean(axis=1, keepdims=True).astype(f32)
    if not keep_emission: m["emission"] = 0.0
    sc["material"] = m
    return sc


def _one_light_scene():
    """BVH_test under the sun sky with exactly one emitter, a sphere whose geometry index equals its BVH-order index"""
    sc = scenes.Scene(scenes.bvh_test_scene(255, hdri=_sun()))
    ps = b2r.PreparedScene(sc, 64, 48)
    i = int(np.nonzero(ps.prim_ids == np.arange(len(ps.prim_ids)))[0][0])
    m = np.ascontiguousarray(sc["material"]).copy(); g = np.ascontiguousarray(sc["geometry"]).copy()
    em = m[int(np.argmax(m["emission"].max(axis=1)))].copy()
    m["emission"] = 0.0
    m = np.concatenate([m, em[None]]).astype(scenes.MATERIAL_DTYPE); g["material_ID"][i] = len(m) - 1
    sc["material"] = m; sc["geometry"] = g
    ps = b2r.PreparedScene(sc, 64, 48)
    assert len(ps.lights) == 1 and ps.lights[0] == i and ps.prim_ids[i] == i
    return sc


BIT_SCENES = {  # name: (scene, product flags, oracle flags, lens)
    "default": (scenes.default_scene, 0, 0, None),
    "bvh_test": (lambda: scenes.bvh_test_scene(255), 0, 0, None),
    "random2000": (lambda: scenes.random_scene(2000, light_every=20), 0, 0, None),
    "ggx_random": (lambda: scenes.ggx_random_scene(400), b2r.FLAG_GGX, ORC_GGX, None),
    "default_glass": (scenes.default_scene, b2r.FLAG_DIELECTRIC, ORC_DIELECTRIC, None),
    "bvh_test_sun_sky": (lambda: scenes.bvh_test_scene(255, hdri=_sun()), b2r.FLAG_SKY_LIGHT, ORC_SKY_LIGHT, None),
    "default_lens": (scenes.default_scene, 0, 0, (0.05, 1.1)),
}


# ------------------------------------------------------------------------------------------------ CPU tier: builder
@pytest.mark.parametrize("case", ["1", "2", "3", "7", "100", "1000", "coincident", "zero_emission"])
def test_builder(case):
    """build_light_tree: every light sits in exactly one leaf, reached by its path bits; each inner box contains its children's boxes and its
    E is the sum of theirs; c and R^2 follow from the box; the build is deterministic; the depth is ceil(log2 n)."""
    n = {"coincident": 9, "zero_emission": 6}.get(case) or int(case)
    lights, lum = _random_lights(n, 3 + n, coincident=case == "coincident", zero=case == "zero_emission")
    prims = np.concatenate([lights[::-1], _random_lights(5, 99)[0]]).astype(scenes.SPHERE_DTYPE)  # every light is a sphere of the scene, in another order
    nodes, light, pl, lo, hi, depth = build(lights, lum, prims)
    assert len(nodes) == 2 * n - 1
    lk = links(nodes)
    leaves = sorted(~lk[lk < 0]); assert leaves == list(range(n))
    inner = np.nonzero(lk >= 0)[0]
    assert (lk[inner] > inner).all()
    for k in inner:
        a, b = lk[k], lk[k] + 1
        for ch in (a, b):
            assert (lo[k] <= lo[ch]).all() and (hi[k] >= hi[ch]).all()
        assert nodes[k, 4] == f32(nodes[a, 4] + nodes[b, 4])
    half = (hi - lo) * f32(0.5)
    assert (nodes[:, :3] == (lo + hi) * f32(0.5)).all()
    assert np.allclose(nodes[:, 3], (half.astype(np.float64) ** 2).sum(axis=1), rtol=1e-6)
    for i in range(n):  # the path bits lead to the light's leaf
        node = 0
        for d in range(light[i, 2]):
            node = lk[node] + ((light[i, 1] >> d) & 1)
        assert lk[node] == ~i and light[i, 3] == node
        assert prims[light[i, 0]].tobytes()[:20] == lights[i].tobytes()[:20]
        assert pl[light[i, 0]] == i
    assert (pl >= 0).sum() == n
    assert depth == (math.ceil(math.log2(n)) if n > 1 else 0) and light[:, 2].max() == depth
    again = build(lights, lum, prims)
    assert all(x.tobytes() == y.tobytes() for x, y in zip((nodes, light, pl, lo, hi), again[:5]))
    if case == "zero_emission":
        assert (nodes[:, 4] == 0).all()


def test_input_rule():
    """light_list_valid: a valid list passes; a light index twice, two lights that are equal spheres, and an emission that is NaN, inf or
    negative are refused."""
    sc = scenes.bvh_test_scene(255); ps = b2r.PreparedScene(sc, 64, 48); L = taps()
    def ok(lights, mat=ps.material, geo=ps.geometry):
        lights = np.ascontiguousarray(lights, np.int32); return L.lt_list_valid(_p(np.ascontiguousarray(mat)), _p(lights), len(lights), _p(np.ascontiguousarray(geo))) == 1
    assert ok(ps.lights) and ok(ps.lights[:0])
    assert not ok(np.r_[ps.lights, ps.lights[2:3]])
    geo = ps.geometry.copy(); extra = int(np.setdiff1d(np.arange(len(geo)), ps.lights)[0]); geo[extra] = geo[ps.lights[0]]
    assert not ok(np.r_[ps.lights, extra], geo=geo)
    for bad in (np.nan, np.inf, -0.5):
        m = ps.material.copy(); m["emission"][ps.geometry["material_ID"][ps.lights[0]], 1] = bad
        assert not ok(ps.lights, mat=m)


# ------------------------------------------------------------------------------------------------ CPU tier: selection pdf and descent
def _tree(n=100, seed=5):
    lights, lum = _random_lights(n, seed)
    nodes, light, pl, lo, hi, depth = build(lights, lum, lights)
    return lights, nodes, light, pl, lo, hi


@pytest.mark.parametrize("n", [1, 2, 100, 1000])
def test_pdf_sums_to_one(n):
    """sum_i light_tree_pdf(P, i) = 1 within 1e-5 for P far away, at every node's centre (inside its box) and on lights' surfaces."""
    lights, nodes, light, pl, lo, hi = _tree(n, 11 + n)
    pts = [np.array([1e5, -3e4, 2e5], f32), np.array([-50, 400, 10], f32)] + list(nodes[:: max(1, len(nodes) // 40), :3])
    r = np.sqrt(lights["radius_sq"]); pos = lights["position"]
    pts += [pos[i] + np.array([r[i], 0, 0], f32) for i in range(0, n, max(1, n // 20))]
    for P in pts:
        assert abs(float(pdf_all(nodes, light, P).astype(np.float64).sum()) - 1.0) <= 1e-5, P


def test_descent_equals_pdf_bit_for_bit():
    """light_tree_pick's accumulated pdf == light_tree_pdf of the picked light, bit for bit, for random (P, u), u = 0, u = 1.0 and u one ulp
    either side of the root's branch threshold (the sum of the left subtree's pdfs)."""
    lights, nodes, light, pl, lo, hi = _tree(300, 2)
    rs = np.random.RandomState(4)
    P = np.concatenate([(rs.rand(400, 3) * [260, 160, 260] - 30).astype(f32), nodes[:50, :3]])
    us = [rs.rand(len(P)).astype(f32), np.zeros(len(P), f32), np.ones(len(P), f32)]
    lk = links(nodes)
    left = np.zeros(len(light), bool)
    stack = [lk[0]]
    while stack:
        k = stack.pop()
        if lk[k] < 0: left[~lk[k]] = True
        else: stack += [lk[k], lk[k] + 1]
    thr = np.array([pdf_all(nodes, light, p)[left].astype(np.float64).sum() for p in P]).astype(f32)
    us += [thr, np.nextafter(thr, f32(0)), np.nextafter(thr, f32(1))]
    for u in us:
        k, pdf, pdf_of = pick(nodes, light, P, u)
        assert pdf.tobytes() == pdf_of.tobytes()
        assert (pdf > 0).all() and (k >= 0).all() and (k < len(light)).all()


def test_descent_chi_square():
    """The leaves the descent picks for uniform u follow the pdf (chi-square over lights with an expected count >= 5, p > 1e-4)."""
    from scipy import stats
    lights, nodes, light, pl, lo, hi = _tree(60, 8)
    for P in (np.array([100, 50, 100], f32), np.array([10, 90, 190], f32)):
        n = 200000
        u = np.random.RandomState(1).rand(n).astype(f32)
        k, _, _ = pick(nodes, light, np.repeat(P[None], n, 0), u)
        e = pdf_all(nodes, light, P).astype(np.float64) * n; c = np.bincount(k, minlength=len(light)).astype(np.float64)
        keep = e >= 5
        obs = np.r_[c[keep], c[~keep].sum()]; exp = np.r_[e[keep], e[~keep].sum()]
        if exp[-1] == 0: obs, exp = obs[:-1], exp[:-1]
        assert stats.chi2.sf(float(((obs - exp) ** 2 / exp).sum()), len(obs) - 1) > 1e-4


@pytest.mark.parametrize("sel_scale", [1.0, 0.5])
def test_mis_complement(sel_scale):
    """For random (P, light, direction): the light sample's selection pdf equals the emissive hit's (bit for bit), so the light-sample weight
    plus the emissive-hit weight of the same direction is 1 within 1e-6 (without a sampled sky: sel_scale 1; with one: 1/2)."""
    lights, nodes, light, pl, lo, hi = _tree(200, 6)
    rs = np.random.RandomState(9); m = 5000
    P = (rs.rand(m, 3) * [220, 120, 220] - 10).astype(f32); u = rs.rand(m).astype(f32)
    k = np.zeros(m, np.int32); a = np.zeros(m, f32); b = np.zeros(m, f32)
    taps().lt_sel_pair(_p(nodes), _p(light), _p(pl), sel_scale, _p(P), _p(u), m, _p(k), _p(a), _p(b))
    assert a.tobytes() == b.tobytes()
    cone = (rs.rand(m) * 50 + 0.1).astype(np.float64); bpdf = (rs.rand(m) / np.pi).astype(np.float64)
    lp = a.astype(np.float64) * cone
    w_l = lp * lp / np.maximum(1e-6, lp * lp + bpdf * bpdf); w_e = bpdf * bpdf / np.maximum(1e-6, bpdf * bpdf + lp * lp)
    ok = lp * lp + bpdf * bpdf >= 1e-6
    assert np.abs(w_l + w_e - 1.0)[ok].max() <= 1e-6


# ------------------------------------------------------------------------------------------------ CPU tier: renderer routines
@pytest.mark.parametrize("name", list(BIT_SCENES))
def test_host_check_equals_the_restatement_bit_for_bit(name):
    """lt_render_sample (the kernels' LTREE shading routines and the host builder's tree, on the host) == the restatement's ORC_LIGHT_TREE
    frames bit for bit: the default scene, BVH_test, a 2000-sphere random scene, ggx_random_scene with GGX, glass, the sun sky with
    B2R_FLAG_SKY_LIGHT, a lens; brute force and the traversal tree; and the frames differ from the flag-off ones."""
    make, pf, of, lens = BIT_SCENES[name]; sc = make(); w, h, mb = 64, 48, 8
    o = LtOracle(w, h, max_bounces=mb, flags=ORC_LIGHT_TREE | of); o.set_scene(sc)
    if lens: o.set_lens(*lens)
    for acc, use_bvh in ((1, 0), (5, 2)):
        ref, _ = o.sample(acc)
        rad = render_taps(sc, w, h, mb, acc, use_bvh, pf, lens)
        assert float(ref.max()) > 0.0
        assert rad.tobytes() == ref.tobytes(), (name, acc, use_bvh)
    o.close()
    if not pf & b2r.FLAG_GGX:
        assert sky_render_taps(sc, w, h, mb, 5, 2, pf, lens).tobytes() != rad.tobytes()


@pytest.mark.parametrize("flags", [0, ORC_SKY_LIGHT])
def test_restatement_without_the_flag_is_the_sky_loop(flags):
    """The restatement without ORC_LIGHT_TREE == the sky restatement's loop, bit for bit (BVH_test under the sun sky)."""
    sc = scenes.bvh_test_scene(255, hdri=_sun()); w, h = 64, 48
    o1 = LtOracle(w, h, max_bounces=8, K=2, flags=flags); o1.set_scene(sc); o1.accumulate(3)
    o2 = SkyOracle(w, h, max_bounces=8, K=2, flags=flags); o2.set_scene(sc); o2.accumulate(3)
    assert o1.buckets().tobytes() == o2.buckets().tobytes()
    o1.close(); o2.close()


@pytest.mark.parametrize("name", ["white_furnace", "bvh_test_dark", "default_sun_dark"])
def test_flag_without_sphere_lights_changes_no_bits(name):
    """With no sphere lights the flag changes no bit: White_Furnace, BVH_test with its emission removed, and the default scene under the sun
    sky with its emission removed (B2R_FLAG_SKY_LIGHT on both sides), on the host check and on the restatement."""
    sc, pf, of = {"white_furnace": (scenes.white_furnace(), 0, 0), "bvh_test_dark": (_gray(scenes.bvh_test_scene(255), False), 0, 0),
                  "default_sun_dark": (_gray(_default_sky(_sun()), False), b2r.FLAG_SKY_LIGHT, ORC_SKY_LIGHT)}[name]
    w, h, mb = 64, 48, 8
    for use_bvh in (0, 2):
        assert render_taps(sc, w, h, mb, 3, use_bvh, pf).tobytes() == sky_render_taps(sc, w, h, mb, 3, use_bvh, pf).tobytes()
    o1 = LtOracle(w, h, max_bounces=mb, K=2, flags=ORC_LIGHT_TREE | of); o1.set_scene(sc); o1.accumulate(3)
    o2 = SkyOracle(w, h, max_bounces=mb, K=2, flags=of); o2.set_scene(sc); o2.accumulate(3)
    assert float(o2.buckets().max()) > 0 and o1.buckets().tobytes() == o2.buckets().tobytes()
    o1.close(); o2.close()


def test_one_light_under_a_sampled_sky_changes_no_bits():
    """One light whose geometry index equals its BVH-order index, under a sampled sky (where quirks Q9 and Q10 already agree with the flag's
    definitions, and a one-leaf tree has pdf 1): flag-on frames == flag-off frames bit for bit, on the host check and the restatement."""
    sc = _one_light_scene(); w, h, mb = 64, 48, 8
    for use_bvh in (0, 2):
        a = render_taps(sc, w, h, mb, 2, use_bvh, b2r.FLAG_SKY_LIGHT); b = sky_render_taps(sc, w, h, mb, 2, use_bvh, b2r.FLAG_SKY_LIGHT)
        assert float(a.max()) > 0 and a.tobytes() == b.tobytes()
    o1 = LtOracle(w, h, max_bounces=mb, K=2, flags=ORC_LIGHT_TREE | ORC_SKY_LIGHT); o1.set_scene(sc); o1.accumulate(3)
    o2 = SkyOracle(w, h, max_bounces=mb, K=2, flags=ORC_SKY_LIGHT); o2.set_scene(sc); o2.accumulate(3)
    assert o1.buckets().tobytes() == o2.buckets().tobytes()
    o1.close(); o2.close()


def _bucket_means(o, n, K):
    o.accumulate(n); b = o.buckets().astype(np.float64)
    return b.mean(axis=(1, 2)) / (n // K)


def test_white_furnace_converges_to_one():
    """White_Furnace with ORC_LIGHT_TREE on the restatement: the frame mean over 16 buckets of 32 samples is 1 within 4 standard errors."""
    K = 16; o = LtOracle(64, 64, max_bounces=4, K=K, flags=ORC_LIGHT_TREE); o.set_scene(scenes.white_furnace())
    m = _bucket_means(o, 32 * K, K); o.close()
    se = m.std(ddof=1) / np.sqrt(K)
    assert abs(m.mean() - 1.0) <= 4 * se + 1e-6, (m.mean(), se)


def _emitter_scene():
    """the default scene, gray and sky-free (three emitters). On the random scenes the light-sampled estimator itself, with or without the
    flag, comes out below MIS-off (DESIGN §2), so they cannot serve as the unbiasedness check of the flag."""
    return _gray(scenes.default_scene())


def test_unbiased_against_no_mis():
    """The default scene, gray and sky-free, max_bounces 32, on the restatement: the flag-on frame mean agrees with the MIS-off mean
    (emission added at every hit, no light sampling: unbiased) within 4 sigma (16 buckets of 24 samples each)."""
    sc = _emitter_scene(); K = 16; out = []
    for fl in (ORC_LIGHT_TREE, ORC_NO_MIS):
        o = LtOracle(64, 48, max_bounces=32, K=K, flags=fl); o.set_scene(sc)
        out.append(_bucket_means(o, 24 * K, K)); o.close()
    a, b = out
    sig = np.sqrt(a.var(ddof=1) / K + b.var(ddof=1) / K)
    assert abs(a.mean() - b.mean()) <= 4 * sig, (a.mean(), b.mean(), sig)


def _pixel_variance(flags, sc, w, h, K, mb):
    o = LtOracle(w, h, max_bounces=mb, K=K, flags=flags | 1); o.set_scene(sc)  # (1 = ORC_BVH: the oracle's stream BVH)
    o.accumulate(K); b = o.buckets().astype(np.float64); o.close()   # [K][3][npix]: one sample per bucket
    return float(b.mean(axis=1).var(axis=0, ddof=1).mean()), float(b.mean())


def test_payoff_variance_at_equal_samples():
    """At equal samples, on a 100k-sphere scene (C3's: 100 emitters) at 48x32, max_bounces 8, 24 samples on the restatement. The two modes
    have different expectations (without the flag quirks Q9 and Q10 bias the sphere lights' estimate low: here the flag-on mean is 1.38x
    the flag-off one), so the per-pixel variance is compared relative to the squared frame mean. Measured: raw variance 1.38x, relative
    variance 0.72x (DESIGN §6); asserted: relative variance below 0.85x."""
    sc = scenes.random_scene(100000); w, h, K, mb = 48, 32, 24, 8
    on, m_on = _pixel_variance(ORC_LIGHT_TREE, sc, w, h, K, mb)
    off, m_off = _pixel_variance(0, sc, w, h, K, mb)
    rel = (on / m_on ** 2) / (off / m_off ** 2)
    print(f"per-pixel variance: flag on {on:.4g}, off {off:.4g}, ratio {on / off:.3f}; means {m_on:.4g} {m_off:.4g}; relative variance ratio {rel:.3f}")
    assert rel < 0.85, (on, off, m_on, m_off)


@pytest.mark.parametrize("other", ["REFERENCE_EXACT", "NO_MIS"])
def test_refused_combinations_at_create(other):
    """B2R_FLAG_LIGHT_TREE with B2R_FLAG_REFERENCE_EXACT or B2R_FLAG_NO_MIS is B2R_ERR_ARG at b2r_create, before a device is needed."""
    cfg = b2r.Config(64, 48, 4, 1, b2r.FLAG_LIGHT_TREE | getattr(b2r, "FLAG_" + other), 0, 0, 0, 0)
    hnd = C.c_void_p(None)
    assert b2r.lib().b2r_create(C.byref(hnd), C.byref(cfg)) == b2r.ERR_ARG
    assert not hnd.value


# ------------------------------------------------------------------------------------------------ GPU tier
def _gpu_vs_restatement(sc, w, h, mb, flags, oflags, lens=None, n=2, **kw):
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags | b2r.FLAG_LIGHT_TREE, **kw)
    o = LtOracle(w, h, max_bounces=mb, flags=ORC_LIGHT_TREE | oflags); o.set_scene(sc)
    if lens: r.SetLens(*lens); o.set_lens(*lens)
    r.Accumulate(n); o.accumulate(n)
    got, want = r.buckets_host(), o.buckets(); r.close(); o.close()
    assert float(want.max()) > 0.0
    return got, want


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("name", list(BIT_SCENES))
@pytest.mark.parametrize("pipe", ["brute", "bvh"])
def test_gpu_equals_the_restatement(name, pipe):
    """Every kernel that shades with the flag (k_bounce_brute FIRST / LENS / later bounces, k_brute_finish, k_shade) == the restatement bit for
    bit on the scenes of the CPU check at 128x96, in both pipelines, across the allowed combinations (GGX, glass, sky light, lens)."""
    make, pf, of, lens = BIT_SCENES[name]
    flags = pf | (b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH)
    got, want = _gpu_vs_restatement(make(), 128, 96, 8, flags, of, lens)
    assert got.tobytes() == want.tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("pipe", ["brute", "bvh"])
def test_gpu_batching_changes_no_bits(pipe):
    """BVH_test with the flag: samples_in_flight 1 without the graph, 2, 16 and 64 (sides and twin lanes) == the restatement; frames enqueued
    back to back == frames waited for."""
    sc = scenes.bvh_test_scene(255); w, h, mb = 128, 96, 8
    flags = (b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH) | b2r.FLAG_LIGHT_TREE
    o = LtOracle(w, h, max_bounces=mb, flags=ORC_LIGHT_TREE); o.set_scene(sc); o.accumulate(64); want = o.buckets(); o.close()
    for extra, spi in ((b2r.FLAG_NO_GRAPH, 1), (0, 2), (0, 16), (0, 64)):
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags | extra, samples_in_flight=spi)
        r.Accumulate(64); got = r.buckets_host(); r.close()
        assert got.tobytes() == want.tobytes(), (extra, spi)
    def frames(wait):
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags)
        for _ in range(6):
            r.Accumulate(1)
            if wait: r.sync(); assert r.Render()
            else: assert r.RenderDevice()
        b = r.buckets_host(); r.close(); return b
    assert frames(False).tobytes() == frames(True).tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("pipe", ["brute", "bvh"])
def test_gpu_context_operations(pipe):
    """b2r_set_flags turning the flag on after an upload == a context created with it (and off again == flag off); a refit then a frame == a
    fresh upload of the moved scene; b2r_read_light_tree == the host builder's output."""
    sc = scenes.random_scene(600, light_every=20); w, h = 128, 96
    base = b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH
    def run(s, flags):
        r = b2r.Renderer(s, w, h, max_bounces=8, buckets=1, flags=flags); r.Accumulate(3); b = r.buckets_host(); r.close(); return b
    want_on, want_off = run(sc, base | b2r.FLAG_LIGHT_TREE), run(sc, base)
    r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=1, flags=base); L = b2r.lib()
    assert L.b2r_set_flags(r._h, base | b2r.FLAG_LIGHT_TREE) == b2r.OK
    r.Accumulate(3); assert r.buckets_host().tobytes() == want_on.tobytes()
    nodes, light_prim = r.read_light_tree()
    hn, hl, hpl = build_ps(r.scene)[:3]
    assert nodes.tobytes() == hn.tobytes() and light_prim.tobytes() == np.ascontiguousarray(hl[:, 0]).tobytes()
    assert L.b2r_set_flags(r._h, base) == b2r.OK
    r.ResetAccumulator(); r.Accumulate(3); assert r.buckets_host().tobytes() == want_off.tobytes()
    r.close()
    geo = sc["geometry"].copy(); rs = np.random.RandomState(3)
    geo["position"] += (rs.uniform(-0.5, 0.5, (len(geo), 3)) * np.sqrt(geo["radius_sq"])[:, None]).astype(f32)
    moved = scenes.Scene(sc); moved["geometry"] = geo
    r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=1, flags=base | b2r.FLAG_LIGHT_TREE)
    r.Accumulate(1); r.RefitScene(geo); r.ResetAccumulator(); r.Accumulate(3)
    got = r.buckets_host(); nodes, light_prim = r.read_light_tree(); hn, hl = build_ps(r.scene)[:2]; r.close()
    assert got.tobytes() == run(moved, base | b2r.FLAG_LIGHT_TREE).tobytes()
    assert nodes.tobytes() == hn.tobytes() and light_prim.tobytes() == np.ascontiguousarray(hl[:, 0]).tobytes()


@pytest.mark.gpu
@needs_gpu
def test_gpu_unbiased_full_size():
    """The default scene, gray and sky-free, at 1920x1088, max_bounces 32, 128 samples in 16 buckets: the flag-on frame mean agrees with the
    MIS-off mean within 4 sigma."""
    sc = _emitter_scene(); K = 16; out = []
    for fl in (b2r.FLAG_LIGHT_TREE, b2r.FLAG_NO_MIS):
        r = b2r.Renderer(sc, 1920, 1088, max_bounces=32, buckets=K, flags=fl | b2r.FLAG_FORCE_BVH)
        r.Accumulate(8 * K); b = r.buckets_host().astype(np.float64); r.close()
        out.append(b.mean(axis=(1, 2)) / 8)
    a, c = out
    sig = np.sqrt(a.var(ddof=1) / K + c.var(ddof=1) / K)
    assert abs(a.mean() - c.mean()) <= 4 * sig, (a.mean(), c.mean(), sig)


@pytest.mark.gpu
@needs_gpu
def test_gpu_flag_rules(tmp_path):
    """The C ABI's rules: each refused combination at b2r_create and at b2r_set_flags; the input rule (a light index twice, a negative
    emission) at upload, refit and b2r_set_flags turning the flag on, accepted without the flag; b2r_read_light_tree without a tree; no
    checkpoint across the flag."""
    sc = scenes.bvh_test_scene(255); L = b2r.lib()
    for other in (b2r.FLAG_REFERENCE_EXACT, b2r.FLAG_NO_MIS):
        with pytest.raises(b2r.B2RError) as e:
            b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_LIGHT_TREE | other)
        assert e.value.code == b2r.ERR_ARG
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=other)
        assert L.b2r_set_flags(r._h, other | b2r.FLAG_LIGHT_TREE) == b2r.ERR_ARG
        r.close()
    dup = b2r.PreparedScene(sc, 64, 48); dup.lights = np.ascontiguousarray(np.r_[dup.lights, dup.lights[:1]], np.int32)
    neg = scenes.Scene(sc); m = np.ascontiguousarray(sc["material"]).copy()
    k = int(sc["geometry"]["material_ID"][dup.lights[0]]); m["emission"][k, 1] = -1.0; neg["material"] = m
    for bad in (dup, neg):
        with pytest.raises(b2r.B2RError) as e:
            b2r.Renderer(bad, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_LIGHT_TREE)
        assert e.value.code == b2r.ERR_ARG
        r = b2r.Renderer(bad, 64, 48, max_bounces=4, buckets=1); r.Accumulate(1)
        assert L.b2r_set_flags(r._h, b2r.FLAG_LIGHT_TREE) == b2r.ERR_ARG
        r.close()
    r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_LIGHT_TREE)
    with pytest.raises(b2r.B2RError) as e:
        r.RefitScene(sc["geometry"], material=m)
    assert e.value.code == b2r.ERR_ARG
    r.close()
    r = b2r.Renderer(scenes.white_furnace(), 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_LIGHT_TREE)
    n = C.c_uint32(0)
    assert L.b2r_read_light_tree(r._h, None, None, C.byref(n)) == b2r.ERR_STATE
    r.close()
    r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1)
    assert L.b2r_read_light_tree(r._h, None, None, C.byref(n)) == b2r.ERR_STATE
    r.close()
    for a, b in ((b2r.FLAG_LIGHT_TREE, 0), (0, b2r.FLAG_LIGHT_TREE)):
        path = tmp_path / f"ck_{a}_{b}.b2r"
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=a); r.Accumulate(2); r.SaveCheckpoint(path); r.close()
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b)
        assert L.b2r_load_checkpoint(r._h, str(path).encode()) == b2r.ERR_STATE
        r.close()
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=a); r.LoadCheckpoint(path); r.close()
