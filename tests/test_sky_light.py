"""The HDRI sky as a light (B2R_FLAG_SKY_LIGHT): light samples drawn from the sky's cell distribution, MIS-combined by the power heuristic with
the BSDF-sampled misses (DESIGN.md §2). The reference samples only its sphere lights, so there is no reference result: the tables and the sampler
are checked against their definition and against float64 integrals, and the kernels bit for bit against the oracle's restatement. That
restatement lives in tests/skycheck/sky_oracle.cpp, which compiles the oracle (unchanged) through the dielectric and lens restatements and adds
the ORC_SKY_LIGHT branches; the product's routines and the tables' host twin run on the CPU through tests/skycheck/sky_taps.cpp. This module
compiles both with g++ into a temporary directory.

CPU tier: tables, sampler, host check against the restatement, unbiasedness on the restatement, the create-time refusals. GPU tier (-m gpu):
every kernel that shades, batching, device tables against the host twin, set_flags after an upload, full-size unbiasedness, the C ABI's rules."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import b2r
import oracle_py
import scenes
from conftest import have_gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
needs_gpu = pytest.mark.skipif(not have_gpu(), reason="needs a CUDA device")
f32 = np.float32
ORC_DIELECTRIC, ORC_SKY_LIGHT = 16, 32

_TAPS = None
_ORACLE = None


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def taps():
    """tests/skycheck/sky_taps.cpp (+ csrc/b2r_host.cpp) with the host check's flags, compiled once per session into a temporary directory"""
    global _TAPS
    if _TAPS is None:
        import tempfile
        csrc = os.path.join(ROOT, "cpu-raytracing-experiments_b200", "csrc")
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_skytaps_"), "libskytaps.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mavx2", "-mfma", "-fPIC", "-shared", "-I/usr/local/cuda/include", "-I", csrc,
                               os.path.join(HERE, "skycheck", "sky_taps.cpp"), os.path.join(csrc, "b2r_host.cpp"), "-o", out])
        L = C.CDLL(out)
        vp, u32 = C.c_void_p, C.c_uint32
        L.sk_build_tables.argtypes = [vp, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp]; L.sk_build_tables.restype = C.c_int
        L.sk_texels_valid.argtypes = [vp, C.c_size_t, vp, vp]; L.sk_texels_valid.restype = C.c_int
        L.sk_sample_dirs.argtypes = [vp, vp, u32, u32, C.c_int32, C.c_int32, vp, u32, vp, vp, vp]; L.sk_sample_dirs.restype = None
        L.sk_row_z.argtypes = [u32, vp]; L.sk_row_z.restype = None
        _TAPS = L
    return _TAPS


def oracle_lib():
    """tests/skycheck/sky_oracle.cpp compiled once per session into a temporary directory (the oracle's flags)"""
    global _ORACLE
    if _ORACLE is None:
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_skycheck_"), "libskycheck.so")
        subprocess.check_call(["g++", "-std=c++17", "-fPIC", "-shared", "-pthread", "-fno-fast-math", "-O2", "-mavx2", "-mfma", "-ffp-contract=off",
                               "-I", os.path.join(ROOT, "oracle"), os.path.join(HERE, "skycheck", "sky_oracle.cpp"), "-o", out])
        L = C.CDLL(out)
        ref = oracle_py.lib()
        for name in ("orc_create", "orc_destroy", "orc_set_scene", "orc_set_camera_lookat", "orc_get_camera_raw", "orc_reset", "orc_set_accumulations",
                     "orc_read_buckets", "orc_render", "orc_read_counters", "orc_reset_counters", "orc_generate_rays"):
            fn, r = getattr(L, name), getattr(ref, name); fn.argtypes = r.argtypes; fn.restype = r.restype
        vp, f = C.c_void_p, C.c_float
        L.dl_accumulate.argtypes = [vp, C.c_uint32, C.c_int]; L.dl_accumulate.restype = None
        L.sk_accumulate.argtypes = [vp, C.c_uint32, C.c_int]; L.sk_accumulate.restype = None
        L.sk_set_tables.argtypes = [vp, vp, vp, vp, C.c_uint32, C.c_uint32]; L.sk_set_tables.restype = None
        L.lo_set_lens.argtypes = [vp, f, f]; L.lo_set_lens.restype = None
        _ORACLE = L
    return _ORACLE


def host_tables(hdri, ambient):
    """the host twin's tables of an [h][w][4] texture: (marg, cond[rows][cols + 1], pdf[h][w], cols, rows)"""
    L = taps(); hdri = np.ascontiguousarray(hdri, f32); h, w = hdri.shape[:2]; amb = np.asarray(ambient, f32)
    cols, rows = C.c_uint32(0), C.c_uint32(0)
    L.sk_build_tables(_p(hdri), w, h, _p(amb), None, None, None, C.byref(cols), C.byref(rows))
    marg = np.empty(rows.value + 1, f32); cond = np.empty((rows.value, cols.value + 1), f32); pdf = np.empty((h, w), f32)
    L.sk_build_tables(_p(hdri), w, h, _p(amb), _p(marg), _p(cond), _p(pdf), C.byref(cols), C.byref(rows))
    return marg, cond, pdf, cols.value, rows.value


def row_z(rows):
    out = np.empty(rows + 1, f32); taps().sk_row_z(rows, _p(out)); return out


def sky_sampled(sc):
    return sc.get("hdri") is not None and max(sc["ambient"]) > 0 and float(np.asarray(sc["hdri"])[..., :3].max()) > 0


class SkyOracle(oracle_py.Oracle):
    """oracle_py.Oracle on the oracle with the sky light restated (flags may hold ORC_SKY_LIGHT, ORC_DIELECTRIC); the host twin's tables"""

    def __init__(self, width, height, max_bounces=16, K=1, flags=0):
        self.L = oracle_lib()
        self.h = self.L.orc_create(width, height, max_bounces, K, flags)
        assert self.h
        self.width, self.height, self.K, self.max_bounces, self.flags = width, height, K, max_bounces, flags
        self.npix = width * height
        self.L.lo_set_lens(self.h, 0.0, 1.0)

    def set_scene(self, sc):
        n = super().set_scene(sc)
        if (self.flags & ORC_SKY_LIGHT) and sky_sampled(sc):
            self._tab = host_tables(sc["hdri"], sc["ambient"]); m, c, p, cols, rows = self._tab
            self.L.sk_set_tables(self.h, _p(m), _p(c), _p(p), cols, rows)
        else:
            self.L.sk_set_tables(self.h, None, None, None, 0, 0)
        return n

    def close(self):
        self.L.sk_set_tables(self.h, None, None, None, 0, 0)
        super().close()

    def accumulate(self, n=1, threads=None):
        self.L.sk_accumulate(self.h, n, threads or os.cpu_count() or 1)

    def set_lens(self, radius, focus_distance):
        self.L.lo_set_lens(self.h, radius, focus_distance)

    def sample(self, acc):
        self.reset(); self.reset_counters(); self.set_accumulations(acc - 1); self.accumulate(1)
        return self.buckets()[0], self.counters()


def render_taps(sc, w, h, mb, acc, use_bvh, flags, lens=None):
    """one sample of every pixel through sk_render_sample (the kernels' shading routines on the host): rad[3][npix] in tile order"""
    ps = b2r.PreparedScene(sc, w, h)
    rad = np.zeros((3, w * h), f32); cnt = (C.c_uint64 * 5)()
    ln = None if lens is None else np.asarray(lens, f32)
    rc = taps().sk_render_sample(_p(ps.prims), _p(ps.nodes), len(ps.prims), len(ps.nodes), _p(ps.material), len(ps.material), _p(ps.lights), len(ps.lights),
                                 _p(ps.geometry), _p(ps.camera), w, h, mb, flags, acc, use_bvh, _p(rad), cnt,
                                 _p(ps.ambient), _p(ps.hdri), 0 if ps.hdri is None else ps.hdri.shape[1], 0 if ps.hdri is None else ps.hdri.shape[0], _p(ln))
    assert rc == 0
    return rad


# ------------------------------------------------------------------------------------------------ scenes
def _gray(sc):
    """the scene with every albedo replaced by its channel mean (quirk Q14 is then moot: tr == tg == tb) and no emitter. Without the flag the
    sphere lights' MIS carries quirks Q9 and Q10 (a biased estimate of the sphere light: measured on BVH_test at 64x48, 384 spp, 1.70 against
    2.00 with MIS off), and the flag takes Q10 out of it, so the two modes agree only where no sphere light is sampled."""
    sc = scenes.Scene(sc); m = np.ascontiguousarray(sc["material"]).copy()
    m["albedo"] = m["albedo"].mean(axis=1, keepdims=True).astype(f32); m["emission"] = 0.0
    sc["material"] = m
    return sc


def _default_sky(hdri=None):
    sc = scenes.Scene(scenes.default_scene()); sc["ambient"] = (0.8, 0.9, 1.0)
    sc["hdri"] = scenes.synthetic_hdri() if hdri is None else hdri
    return sc


def _sun(w=128, h=64):
    return scenes.sun_hdri(w, h, sun_radius_deg=6.0, sun_radiance=200.0)


def _furnace_sun():
    sc = scenes.Scene(scenes.white_furnace()); sc["hdri"] = _sun(); sc["ambient"] = (1.0, 0.5, 0.25)
    return sc


BIT_SCENES = {  # name: (scene, extra product flags, oracle flags, lens)
    "bvh_test": (lambda: scenes.bvh_test_scene(255), 0, 0, None),
    "bvh_test_sun": (lambda: scenes.bvh_test_scene(255, hdri=_sun()), 0, 0, None),
    "white_furnace": (scenes.white_furnace, 0, 0, None),
    "white_furnace_sun": (_furnace_sun, 0, 0, None),
    "brdf_test": (scenes.brdf_test_scene, 0, 0, None),
    "default_sky_lens": (_default_sky, 0, 0, (0.05, 1.1)),
    "default_sky_glass": (lambda: _default_sky(_sun()), b2r.FLAG_DIELECTRIC, ORC_DIELECTRIC, None),
}


def _textures():
    rs = np.random.RandomState(7)
    def rnd(h, w):
        t = np.ones((h, w, 4), f32); t[..., :3] = rs.rand(h, w, 3).astype(f32) * f32(3.0); return t
    return {"synthetic": scenes.synthetic_hdri(), "sun": _sun(256, 128), "1x1": np.ones((1, 1, 4), f32), "1xN": rnd(9, 1), "Nx1": rnd(1, 11),
            "2x2": rnd(2, 2), "dark_rows": np.concatenate([np.zeros((5, 16, 4), f32), rnd(4, 16)])}


# ------------------------------------------------------------------------------------------------ CPU tier: tables and sampler
@pytest.mark.parametrize("name", list(_textures()))
def test_tables_are_distributions(name):
    """The host twin's tables: both CDFs start at 0, end at exactly 1 and increase strictly (every cell has a non-zero probability); the cell
    pdfs integrate to 1 over the cells' solid angles (sum pdf_c * Omega_c, in float64, within a few ulps per cell); the texture's last column
    and row repeat the adjacent cell's pdf; the pdf is positive and finite everywhere."""
    tex = _textures()[name]; amb = (1.0, 0.7, 0.4)
    marg, cond, pdf, cols, rows = host_tables(tex, amb)
    h, w = tex.shape[:2]
    assert cols == max(w - 1, 1) and rows == max(h - 1, 1)
    for cdf in [marg] + list(cond):
        assert cdf[0] == 0.0 and cdf[-1] == 1.0 and (np.diff(cdf.astype(np.float64)) > 0).all()
    z = row_z(rows).astype(np.float64)
    assert z[0] == 1.0 and z[-1] == -1.0 and (np.diff(z) < 0).all()
    omega = (2 * np.pi / cols) * (z[:-1] - z[1:])
    cell_pdf = pdf[:rows, :cols].astype(np.float64)
    assert np.isfinite(pdf).all() and (pdf > 0).all()
    total = float((cell_pdf * omega[:, None]).sum())
    assert abs(total - 1.0) <= 8 * 2.0 ** -24 * np.sqrt(cols * rows) + 1e-6, total
    if w > 1: assert (pdf[:, w - 1] == pdf[:, w - 2]).all()
    if h > 1: assert (pdf[h - 1, :] == pdf[h - 2, :]).all()
    p_cell = np.diff(marg.astype(np.float64))[:, None] * np.diff(cond.astype(np.float64), axis=1)
    assert np.allclose(cell_pdf * omega[:, None], p_cell, rtol=1e-6, atol=0)


def test_zero_sky_input_rule():
    """sky_texels_valid: finite, non-negative texels pass; a NaN, an inf or a negative value fails in a channel whose ambient is > 0 and is
    ignored in one whose ambient is 0; a texture that is zero everywhere passes and is flagged as not sampled."""
    L = taps(); nz = C.c_int(0)
    def check(tex, amb):
        tex = np.ascontiguousarray(tex, f32); return L.sk_texels_valid(_p(tex), tex.shape[0] * tex.shape[1], _p(np.asarray(amb, f32)), C.byref(nz)), nz.value
    base = scenes.synthetic_hdri()
    assert check(base, (1, 1, 1)) == (1, 1)
    assert check(np.zeros((4, 4, 4), f32), (1, 1, 1)) == (1, 0)
    for bad in (np.nan, np.inf, -0.5):
        t = base.copy(); t[3, 5, 1] = bad
        assert check(t, (1, 1, 1))[0] == 0
        assert check(t, (1, 0, 1))[0] == 1
        t = base.copy(); t[3, 5, 3] = bad   # the alpha channel is never read
        assert check(t, (1, 1, 1))[0] == 1


def _draw(tab, tex, n, seed):
    marg, cond, pdf, cols, rows = tab; h, w = tex.shape[:2]
    u = np.random.RandomState(seed).rand(n, 4).astype(f32)
    dirs = np.empty((n, 3), f32); cells = np.empty(n, np.int32); texels = np.empty(n, np.int32)
    taps().sk_sample_dirs(_p(marg), _p(np.ascontiguousarray(cond)), cols, rows, w, h, _p(u), n, _p(dirs), _p(cells), _p(texels))
    return u, dirs, cells, texels


@pytest.mark.parametrize("name", ["synthetic", "sun", "1x1", "1xN", "Nx1"])
def test_sampler(name):
    """sky_sample_dir: the histogram of drawn cells matches the cell probabilities (chi-square over cells with an expected count >= 5, p > 1e-4);
    every direction lies in its drawn cell by the exact mapping (longitude and dy against the cell's borders, float64, a few ulps); the
    polynomial lookup (sky_texel) returns the drawn cell's texel except within 1e-4 rad of a border."""
    from scipy import stats
    tex = _textures()[name]; tab = host_tables(tex, (1, 1, 1)); marg, cond, pdf, cols, rows = tab; w = tex.shape[1]
    n = 200000
    u, dirs, cells, texels = _draw(tab, tex, n, 11)
    j, i = cells // w, cells % w
    assert (i < cols).all() and (j < rows).all()
    p_cell = (np.diff(marg.astype(np.float64))[:, None] * np.diff(cond.astype(np.float64), axis=1)).ravel()
    counts = np.bincount(j * cols + i, minlength=cols * rows).astype(np.float64)
    e = p_cell * n; keep = e >= 5
    if keep.sum() > 1:
        obs = np.r_[counts[keep], counts[~keep].sum()]; exp = np.r_[e[keep], e[~keep].sum()]
        if exp[-1] == 0: obs, exp = obs[:-1], exp[:-1]
        chi2 = float(((obs - exp) ** 2 / exp).sum())
        assert stats.chi2.sf(chi2, len(obs) - 1) > 1e-4, chi2
    d = dirs.astype(np.float64)
    z = row_z(rows).astype(np.float64)
    eps = 1e-6
    assert ((d[:, 1] <= z[j] + eps) & (d[:, 1] >= z[j + 1] - eps)).all()
    lon = np.arctan2(d[:, 2], d[:, 0]); lo = 2 * np.pi * i / cols - np.pi; hi = 2 * np.pi * (i + 1) / cols - np.pi
    dl = np.minimum(np.abs(lon - lo), np.abs(lon - hi))
    inside = (lon >= lo - 1e-5) & (lon <= hi + 1e-5)
    if cols > 1: assert inside.all()
    assert (np.abs(np.linalg.norm(d, axis=1) - 1.0) < 1e-5).all()
    lat = np.arcsin(np.clip(d[:, 1], -1, 1)); zlat = np.arcsin(np.clip(z, -1, 1))
    near = (cols > 1) & (dl < 1e-4) | (np.minimum(np.abs(lat - zlat[j]), np.abs(lat - zlat[j + 1])) < 1e-4) & (rows > 1)
    tx_i, tx_j = texels % w, texels // w
    agree = (np.minimum(tx_i, cols - 1) == i) & (np.minimum(tx_j, rows - 1) == j)
    assert (agree | near).all(), int((~agree & ~near).sum())


@pytest.mark.parametrize("name", ["synthetic", "sun"])
def test_sampler_estimates_the_irradiance(name):
    """Monte Carlo integral of L(d) max(cos, 0) / pdf over sky samples (normal +y and a tilted one; L and the pdf by the lookup, as the
    renderer evaluates them) matches a float64 quadrature of the texture over the lookup's texels (4096 x 2048 midpoints) within 5 sigma."""
    tex = _textures()[name]; tab = host_tables(tex, (1, 1, 1)); marg, cond, pdf, cols, rows = tab; h, w = tex.shape[:2]
    n = 400000
    u, dirs, cells, texels = _draw(tab, tex, n, 5)
    lum = tex[..., :3].astype(np.float64).mean(axis=2).ravel()
    pdf_drawn = pdf.ravel()[cells].astype(np.float64)
    qa, qb = 4096, 2048
    lon = (np.arange(qa) + 0.5) / qa * 2 * np.pi - np.pi; lat = np.pi / 2 - (np.arange(qb) + 0.5) / qb * np.pi
    dy = np.sin(lat)[:, None]; r = np.cos(lat)[:, None]; dx = r * np.cos(lon)[None, :]; dz = r * np.sin(lon)[None, :]
    uu = (w - 1) * (0.5 + np.arctan2(dz, dx) / (2 * np.pi)); vv = (h - 1) * (0.5 - np.arcsin(np.broadcast_to(dy, dx.shape)) / np.pi)
    tq = vv.astype(np.int64) * w + uu.astype(np.int64)
    dA = (2 * np.pi / qa) * (np.pi / qb) * np.cos(lat)[:, None]
    for nrm in (np.array([0.0, 1.0, 0.0]), np.array([0.6, 0.3, -0.74]) / np.linalg.norm([0.6, 0.3, -0.74])):
        cosq = np.maximum(dx * nrm[0] + dy * nrm[1] + dz * nrm[2], 0.0)
        exact = float((lum[tq] * cosq * dA).sum())
        c = np.maximum(dirs.astype(np.float64) @ nrm, 0.0)
        x = lum[texels] * c / pdf_drawn
        assert abs(x.mean() - exact) <= 5 * x.std() / np.sqrt(n) + 2e-3 * exact, (x.mean(), exact)


# ------------------------------------------------------------------------------------------------ CPU tier: renderer routines
@pytest.mark.parametrize("name", list(BIT_SCENES))
def test_host_check_equals_the_restatement_bit_for_bit(name):
    """sk_render_sample with the flag (the kernels' shading routines and the host twin's tables, on the host) == the restatement's
    ORC_SKY_LIGHT frames bit for bit: BVH_test (synthetic and sun sky), White_Furnace (its 1x1 sky, and a sun sky), BRDF_test, the default
    scene under a sky with a lens and with glass; brute force and the traversal tree; and the frames differ from the flag-off ones."""
    make, pf, of, lens = BIT_SCENES[name]; sc = make(); w, h, mb = 64, 48, 8
    o = SkyOracle(w, h, max_bounces=mb, flags=ORC_SKY_LIGHT | of); o.set_scene(sc)
    if lens: o.set_lens(*lens)
    for acc, use_bvh in ((1, 0), (5, 2)):
        ref, _ = o.sample(acc)
        rad = render_taps(sc, w, h, mb, acc, use_bvh, b2r.FLAG_SKY_LIGHT | pf, lens)
        assert float(ref.max()) > 0.0
        assert rad.tobytes() == ref.tobytes(), (name, acc, use_bvh)
        off = render_taps(sc, w, h, mb, acc, use_bvh, pf, lens)
        assert off.tobytes() != rad.tobytes()
    o.close()


@pytest.mark.parametrize("name", ["default", "random"])
def test_flag_without_a_sky_changes_no_bits(name):
    """Flag on over a scene without a sky (ambient 0; and a sky that is zero everywhere) == flag off, bit for bit, on the host check and on the
    restatement; and the restatement without ORC_SKY_LIGHT is the dielectric restatement's loop."""
    sc = scenes.default_scene() if name == "default" else scenes.random_scene(300, light_every=20)
    w, h, mb = 64, 48, 8
    zero = scenes.Scene(sc); zero["ambient"] = (1.0, 1.0, 1.0); zero["hdri"] = np.zeros((8, 16, 4), f32)
    for s in (sc, zero):
        for use_bvh in (0, 2):
            a = render_taps(s, w, h, mb, 3, use_bvh, b2r.FLAG_SKY_LIGHT); b = render_taps(s, w, h, mb, 3, use_bvh, 0)
            assert a.tobytes() == b.tobytes(), (s is zero, use_bvh)
        o1 = SkyOracle(w, h, max_bounces=mb, K=2, flags=ORC_SKY_LIGHT); o1.set_scene(s); o1.accumulate(3)
        o2 = SkyOracle(w, h, max_bounces=mb, K=2, flags=0); o2.set_scene(s); o2.L.dl_accumulate(o2.h, 3, os.cpu_count() or 1)
        o3 = SkyOracle(w, h, max_bounces=mb, K=2, flags=0); o3.set_scene(s); o3.accumulate(3)
        assert o1.buckets().tobytes() == o2.buckets().tobytes(), s is zero
        assert o3.buckets().tobytes() == o2.buckets().tobytes()
        for o in (o1, o2, o3): o.close()


def _bucket_means(o, n, K):
    o.accumulate(n); b = o.buckets().astype(np.float64)   # [K][3][npix], each bucket the sum of n / K samples
    return b.mean(axis=(1, 2)) / (n // K)


def test_white_furnace_converges_to_ambient():
    """White_Furnace with the flag on the restatement: every pixel's expected linear value is the ambient 1; the frame mean over 16 buckets of
    32 samples is 1 within 4 standard errors, and pixels whose camera ray misses the sphere are exactly 1."""
    sc = scenes.white_furnace(); w = h = 64; K = 16
    o = SkyOracle(w, h, max_bounces=4, K=K, flags=ORC_SKY_LIGHT); o.set_scene(sc)
    m = _bucket_means(o, 32 * K, K); o.close()
    se = m.std(ddof=1) / np.sqrt(K)
    assert abs(m.mean() - 1.0) <= 4 * se + 1e-6, (m.mean(), se)
    assert se > 0


def _gray_means(mb, K=16, spp=24):
    """frame means per bucket of gray, emitter-free BVH_test under synthetic_hdri at 64x48 on the restatement, with and without the flag"""
    sc = _gray(scenes.bvh_test_scene(255)); out = []
    for fl in (ORC_SKY_LIGHT, 0):
        o = SkyOracle(64, 48, max_bounces=mb, K=K, flags=fl); o.set_scene(sc)
        out.append(_bucket_means(o, spp * K, K)); o.close()
    a, b = out
    return a.mean(), b.mean(), np.sqrt(a.var(ddof=1) / K + b.var(ddof=1) / K)


def test_flag_on_and_off_agree_on_a_gray_scene():
    """BVH_test with gray albedos and no emitter under synthetic_hdri, restatement, max_bounces 32 (where quirk Q11 drops a negligible share
    of the energy): frame means with and without the flag agree within 4 sigma (16 buckets of 24 samples each)."""
    a, b, sig = _gray_means(32)
    assert abs(a - b) <= 4 * sig, (a, b, sig)


def test_last_bounce_drop_takes_the_sky_samples_too():
    """Quirk Q11 zeroes the radiance of a path that still hits at the last bounce. With the flag that radiance includes the sky's light samples
    of its earlier bounces, while without it the sky arrives only at a miss, which ends the path: at a small max_bounces the flag-on mean is
    lower by more than 4 sigma (DESIGN §2). Same scene as above, max_bounces 3."""
    a, b, sig = _gray_means(3)
    assert b - a > 4 * sig, (a, b, sig)


@pytest.mark.parametrize("other", ["REFERENCE_EXACT", "NO_MIS", "GGX"])
def test_refused_combinations_at_create(other):
    """B2R_FLAG_SKY_LIGHT with B2R_FLAG_REFERENCE_EXACT, B2R_FLAG_NO_MIS or B2R_FLAG_GGX is B2R_ERR_ARG at b2r_create, before a device is needed."""
    cfg = b2r.Config(64, 48, 4, 1, b2r.FLAG_SKY_LIGHT | getattr(b2r, "FLAG_" + other), 0, 0, 0, 0)
    hnd = C.c_void_p(None)
    assert b2r.lib().b2r_create(C.byref(hnd), C.byref(cfg)) == b2r.ERR_ARG
    assert not hnd.value


# ------------------------------------------------------------------------------------------------ GPU tier
def _gpu_vs_restatement(sc, w, h, mb, flags, oflags, lens=None, n=2, **kw):
    r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags | b2r.FLAG_SKY_LIGHT, **kw)
    o = SkyOracle(w, h, max_bounces=mb, flags=ORC_SKY_LIGHT | oflags); o.set_scene(sc)
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
    bit on the scenes of the CPU check at 128x96, in both pipelines."""
    make, pf, of, lens = BIT_SCENES[name]
    flags = pf | (b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH)
    got, want = _gpu_vs_restatement(make(), 128, 96, 8, flags, of, lens)
    assert got.tobytes() == want.tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("pipe", ["brute", "bvh"])
def test_gpu_batching_changes_no_bits(pipe):
    """BVH_test under the sun sky with the flag: samples_in_flight 1 without the graph, 2 and 16 (sides and twin lanes) == the restatement;
    frames enqueued back to back == frames waited for; the brute-force hand-over to k_brute_finish is exercised (B2R default threshold)."""
    sc = scenes.bvh_test_scene(255, hdri=_sun()); w, h, mb = 128, 96, 8
    flags = b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH
    o = SkyOracle(w, h, max_bounces=mb, flags=ORC_SKY_LIGHT); o.set_scene(sc); o.accumulate(16); want = o.buckets(); o.close()
    for extra, spi in ((b2r.FLAG_NO_GRAPH, 1), (0, 2), (0, 16)):
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags | extra | b2r.FLAG_SKY_LIGHT, samples_in_flight=spi)
        r.Accumulate(16); got = r.buckets_host(); r.close()
        assert got.tobytes() == want.tobytes(), (extra, spi)
    def frames(wait):
        r = b2r.Renderer(sc, w, h, max_bounces=mb, buckets=1, flags=flags | b2r.FLAG_SKY_LIGHT)
        for _ in range(6):
            r.Accumulate(1)
            if wait: r.sync(); assert r.Render()
            else: assert r.RenderDevice()
        b = r.buckets_host(); r.close(); return b
    assert frames(False).tobytes() == frames(True).tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("size", [(64, 32), (1, 1), (1, 9), (11, 1), (2048, 1024), (8192, 4096)])
def test_gpu_tables_equal_the_host_twin(size):
    """The tables k_sky_* build from the device copy of the texture (b2r_read_sky_tables) == the host twin bit for bit, up to 8192 x 4096."""
    w, h = size
    tex = scenes.sun_hdri(w, h) if w * h >= 64 else (np.random.RandomState(w * 31 + h).rand(h, w, 4).astype(f32) + f32(0.1))
    sc = scenes.Scene(scenes.white_furnace()); sc["hdri"] = tex; sc["ambient"] = (1.0, 0.8, 0.6)
    r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_SKY_LIGHT)
    marg, cond, pdf = r.read_sky_tables(); r.close()
    m2, c2, p2, cols, rows = host_tables(tex, sc["ambient"])
    assert marg.tobytes() == m2.tobytes() and cond.tobytes() == c2.tobytes() and pdf.tobytes() == p2.tobytes()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("pipe", ["brute", "bvh"])
def test_gpu_set_flags_after_upload_equals_create(pipe):
    """Turning the flag on with b2r_set_flags after an upload without it (tables built from the device copy) gives the frames of a context
    created with the flag; turning it off again gives the flag-off frames."""
    sc = scenes.bvh_test_scene(255, hdri=_sun()); w, h = 128, 96
    base = b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH
    def run(flags):
        r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=1, flags=flags); r.Accumulate(3); b = r.buckets_host(); r.close(); return b
    want_on, want_off = run(base | b2r.FLAG_SKY_LIGHT), run(base)
    r = b2r.Renderer(sc, w, h, max_bounces=8, buckets=1, flags=base); L = b2r.lib()
    assert L.b2r_set_flags(r._h, base | b2r.FLAG_SKY_LIGHT) == b2r.OK
    r.Accumulate(3); assert r.buckets_host().tobytes() == want_on.tobytes()
    assert L.b2r_set_flags(r._h, base) == b2r.OK
    r.ResetAccumulator(); r.Accumulate(3); assert r.buckets_host().tobytes() == want_off.tobytes()
    r.close()


@pytest.mark.gpu
@needs_gpu
def test_gpu_white_furnace_full_size():
    """White_Furnace at 1920x1088 with the flag, 64 samples in 16 buckets: the frame mean is 1 within 4 standard errors."""
    sc = scenes.white_furnace(); K = 16
    r = b2r.Renderer(sc, 1920, 1088, max_bounces=4, buckets=K, flags=b2r.FLAG_SKY_LIGHT)
    r.Accumulate(4 * K); b = r.buckets_host().astype(np.float64); r.close()
    m = b.mean(axis=(1, 2)) / 4; se = m.std(ddof=1) / np.sqrt(K)
    assert abs(m.mean() - 1.0) <= 4 * se + 1e-6, (m.mean(), se)


@pytest.mark.gpu
@needs_gpu
def test_gpu_flag_on_and_off_agree_full_size():
    """BVH_test with gray albedos and no emitter under synthetic_hdri at 1920x1088, 128 samples in 16 buckets, max_bounces 32 (at 8, quirk
    Q11's drop of the flag's sky samples at the last bounce shows: DESIGN §2): frame means with and without the flag agree within 4 sigma."""
    sc = _gray(scenes.bvh_test_scene(255)); K = 16
    out = []
    for fl in (b2r.FLAG_SKY_LIGHT, 0):
        r = b2r.Renderer(sc, 1920, 1088, max_bounces=32, buckets=K, flags=fl | b2r.FLAG_FORCE_BVH)
        r.Accumulate(8 * K); b = r.buckets_host().astype(np.float64); r.close()
        out.append(b.mean(axis=(1, 2)) / 8)
    a, c = out
    sig = np.sqrt(a.var(ddof=1) / K + c.var(ddof=1) / K)
    assert abs(a.mean() - c.mean()) <= 4 * sig, (a.mean(), c.mean(), sig)


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("pipe", ["brute", "bvh"])
def test_gpu_flag_without_a_sky_changes_no_bits(pipe):
    """On the GPU too: the flag over a scene without a sky (the default scene, ambient 0) and over a sky that is zero everywhere gives the
    frames of the flag off, bit for bit."""
    sc = scenes.default_scene(); zero = scenes.Scene(sc); zero["ambient"] = (1.0, 1.0, 1.0); zero["hdri"] = np.zeros((8, 16, 4), f32)
    base = b2r.FLAG_FORCE_BRUTE if pipe == "brute" else b2r.FLAG_FORCE_BVH
    for s in (sc, zero):
        out = []
        for fl in (base, base | b2r.FLAG_SKY_LIGHT):
            r = b2r.Renderer(s, 128, 96, max_bounces=8, buckets=2, flags=fl); r.Accumulate(4); out.append(r.buckets_host()); r.close()
        assert float(out[0].max()) > 0.0 and out[0].tobytes() == out[1].tobytes()


@pytest.mark.gpu
@needs_gpu
def test_gpu_flag_rules(tmp_path):
    """The C ABI's rules: each refused combination at b2r_create and at b2r_set_flags (flags unchanged); a bad sky texel under the flag at
    upload and at b2r_set_flags turning the flag on, accepted without it; b2r_read_sky_tables without tables; no checkpoint across the flag."""
    sc = scenes.bvh_test_scene(255); L = b2r.lib()
    for other in (b2r.FLAG_REFERENCE_EXACT, b2r.FLAG_NO_MIS, b2r.FLAG_GGX):
        with pytest.raises(b2r.B2RError) as e:
            b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_SKY_LIGHT | other)
        assert e.value.code == b2r.ERR_ARG
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=other)
        assert L.b2r_set_flags(r._h, other | b2r.FLAG_SKY_LIGHT) == b2r.ERR_ARG
        r.close()
    for bad in (np.nan, np.inf, -1.0):
        s = scenes.Scene(sc); t = s["hdri"].copy(); t[5, 7, 2] = bad; s["hdri"] = t
        with pytest.raises(b2r.B2RError) as e:
            b2r.Renderer(s, 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_SKY_LIGHT)
        assert e.value.code == b2r.ERR_ARG
        r = b2r.Renderer(s, 64, 48, max_bounces=4, buckets=1); r.Accumulate(1)
        assert L.b2r_set_flags(r._h, b2r.FLAG_SKY_LIGHT) == b2r.ERR_ARG
        r.close()
    r = b2r.Renderer(scenes.default_scene(), 64, 48, max_bounces=4, buckets=1, flags=b2r.FLAG_SKY_LIGHT)
    cols, rows = C.c_uint32(0), C.c_uint32(0)
    assert L.b2r_read_sky_tables(r._h, None, None, None, C.byref(cols), C.byref(rows)) == b2r.ERR_STATE
    r.close()
    for a, b in ((b2r.FLAG_SKY_LIGHT, 0), (0, b2r.FLAG_SKY_LIGHT)):
        path = tmp_path / f"ck_{a}_{b}.b2r"
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=a); r.Accumulate(2); r.SaveCheckpoint(path); r.close()
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=b)
        assert L.b2r_load_checkpoint(r._h, str(path).encode()) == b2r.ERR_STATE
        r.close()
        r = b2r.Renderer(sc, 64, 48, max_bounces=4, buckets=1, flags=a); r.LoadCheckpoint(path); r.close()
