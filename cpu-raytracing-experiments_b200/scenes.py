"""Scene + camera inputs, as plain numpy records layout-identical to the reference PODs.

Sphere   (32 B)  Primitives.hpp:7-17     {vec3 position; float radius_sq; int32 material_ID} alignas(16)
Material (96 B)  Primitives.hpp:18-27    {albedo, F0, F80, emission, transmission; roughness; IOR_minus_one} alignas(32)
Node     (32 B)  BVH.hpp:18-27           {vec3 min; u32 first_id; vec3 max; u32 prim_count}

`default_scene()` is Scenes::Default verbatim (Application.cpp:33-101); `random_scene(n)` is the BVH_test
distribution (Application.cpp:107-121) drawn with the reference's own PCG (Random.hpp) as SURVEY.md §8d C3
prescribes (std:: distributions are not portable); `white_furnace()` is Application.cpp:218-223.
The same arrays are fed to the CUDA library and to the oracle, so both see bit-identical inputs.
"""
import numpy as np

SPHERE_DTYPE = np.dtype({"names": ["position", "radius_sq", "material_ID"],
                         "formats": [("<f4", 3), "<f4", "<i4"], "offsets": [0, 12, 16], "itemsize": 32})
MATERIAL_DTYPE = np.dtype({"names": ["albedo", "F0", "F80", "emission", "transmission", "roughness", "IOR_minus_one"],
                           "formats": [("<f4", 3)] * 5 + ["<f4", "<f4"], "offsets": [0, 12, 24, 36, 48, 60, 64], "itemsize": 96})
NODE_DTYPE = np.dtype({"names": ["min_bound", "first_id", "max_bound", "prim_count"],
                       "formats": [("<f4", 3), "<u4", ("<f4", 3), "<u4"], "offsets": [0, 12, 16, 28], "itemsize": 32})

f32 = np.float32


def _mat(**kw):
    m = np.zeros((), dtype=MATERIAL_DTYPE)  # Material{} value-initialises to zero
    for k, v in kw.items():
        m[k] = np.asarray(v, dtype=np.float64).astype(np.float32)
    return m


def _sphere(pos, r2, mat):
    s = np.zeros((), dtype=SPHERE_DTYPE)
    s["position"] = np.asarray(pos, dtype=np.float64).astype(np.float32)
    s["radius_sq"] = f32(r2)
    s["material_ID"] = mat
    return s


class Scene(dict):
    """geometry, material, camera{eye,dir,focal_length,exposure}, ambient, hdri (H,W,4 float32 or None)."""
    __getattr__ = dict.__getitem__


def default_scene():
    """Scenes::Default, Application.cpp:33-101 (9 spheres, 9 materials, 3 emissive, ambient 0)."""
    mats, geo = [], []

    def add(pos, r2, **kw):
        mats.append(_mat(**kw))
        geo.append(_sphere(pos, r2, len(mats) - 1))

    r15 = f32(1.5) * f32(1.5); r005 = f32(0.05) * f32(0.05)
    add((0.3, -1.47, 0.0), r15, albedo=[1, 1, 1], F0=[0.8] * 3, F80=[0.9] * 3, roughness=f32(0.2))
    add((0.29999, 0.0801, 0.0), r005, emission=(f32(0.1) * np.array([25, 25, 200], f32)), albedo=[1] * 3, roughness=1.0)
    add((0.3302, 0.36165, 0.7119), r005, emission=(f32(0.1) * np.array([150, 150, 150], f32)), albedo=[1] * 3, roughness=1.0)
    add((-0.4857, -0.0242, -0.41383), r005, emission=[200, 17, 25], albedo=[1] * 3, roughness=1.0)
    add((0.3, 1.7, 0.0), r15, albedo=[0.793, 0.793, 0.664], F0=[0.04] * 3, F80=[0.5] * 3, roughness=f32(0.85))
    add((0.018, f32(0.022), 0.07), f32(0.02) * f32(0.02), albedo=[f32(0.05)] * 3, F0=[f32(0.03)] * 3, F80=[0.5] * 3,
        transmission=[0.95] * 3, IOR_minus_one=f32(0.44), roughness=0.05)
    add((-0.037, f32(0.022), 0.0), f32(0.03) * f32(0.03), albedo=[1] * 3, F0=[0.944, 0.776, 0.373], F80=[f32(0.8), f32(0.8), f32(0.6)], roughness=0.15)
    add((-0.0846, -0.0334, 0.283), f32(0.012) * f32(0.012), albedo=[1] * 3, F0=[0.076288, 0.077375, 0.078887], F80=[0.47990, 0.48028, 0.48080],
        transmission=[0.670, 0.764, 0.855], IOR_minus_one=f32(0.762), roughness=0.1)
    add((0.03863, -0.00788, 0.2835), f32(0.012) * f32(0.012), albedo=[1] * 3, F0=[0.04] * 3, F80=[0.5] * 3, roughness=f32(0.8))
    return Scene(name="default", geometry=np.array(geo, dtype=SPHERE_DTYPE), material=np.array(mats, dtype=MATERIAL_DTYPE),
                 camera=dict(eye=(-0.2, 0.3, 1.0), dir=(0.1, -0.4, -1.0), focal_length=40.0, exposure=1.0),
                 ambient=(0.0, 0.0, 0.0), hdri=None)


def white_furnace():
    """Scenes::White_Furnace, Application.cpp:218-223, with a 1x1 white HDRI (known answer: every linear pixel == ambient)."""
    mats = [_mat(albedo=[1, 1, 1])]
    geo = [_sphere((0, 0, 0), 1.0, 0)]
    return Scene(name="white_furnace", geometry=np.array(geo, dtype=SPHERE_DTYPE), material=np.array(mats, dtype=MATERIAL_DTYPE),
                 camera=dict(eye=(0, 0, 3), dir=(0, 0, -1), focal_length=50.0, exposure=1.0),
                 ambient=(1.0, 1.0, 1.0), hdri=np.ones((1, 1, 4), np.float32))


def brdf_test_scene(hdri=None, gradations=10):
    """Scenes::BRDF_test, Application.cpp:123-217, in the variant the source selects (`switch (Properties::Roughness)`): a dark floor
    sphere, one spherical light of emission 100, and a row of `gradations` unit spheres whose roughness runs 0..1 with F0 = F80 = 1 and
    ALBEDO 0 — under the shipped Lambertian closure (BRDF 0, Renderer.hpp:70) they are black bodies: throughput drops to 0 at the first
    hit and Russian roulette sees q = 1 (Q13). Ambient (1,1,1) over an HDRI sky; camera {0, 0, 2.8 * gradations} -> -z."""
    mats, geo = [], []
    mats.append(_mat(albedo=[f32(0.1)] * 3, roughness=1.0)); geo.append(_sphere((0.0, -1001.0, 0.0), f32(1000.0) * f32(1000.0), 0))
    mats.append(_mat(emission=[100.0, 100.0, 100.0])); geo.append(_sphere((0.0, 10.0, 0.0), 5.0, 1))
    for i in range(gradations):
        t = f32(i) / f32(gradations - 1)
        x = f32(i * 2 - gradations) * f32(1.25) + f32(1.0)
        mats.append(_mat(F0=[1, 1, 1], F80=[1, 1, 1], albedo=[0, 0, 0], roughness=t))
        geo.append(_sphere((x, f32(i) * f32(0.1), 0.0), 1.0, len(mats) - 1))
    return Scene(name="brdf_test", geometry=np.array(geo, dtype=SPHERE_DTYPE), material=np.array(mats, dtype=MATERIAL_DTYPE),
                 camera=dict(eye=(0.0, 0.0, float(f32(gradations) * f32(2.8))), dir=(0, 0, -1), focal_length=50.0, exposure=1.0),
                 ambient=(1.0, 1.0, 1.0), hdri=synthetic_hdri() if hdri is None else hdri)


# ---- the reference's PCG (Random.hpp:5-29), vectorised: state_k = A^k s0 + C (A^k - 1)/(A - 1)  (mod 2^32)
_A = np.uint32(747796405); _C = np.uint32(2891336453)


def _hash_u32(i):
    i = np.uint32(i)
    with np.errstate(over="ignore"):
        i ^= i >> np.uint32(16); i = np.uint32(i * np.uint32(0x21F0AAAD)); i ^= i >> np.uint32(15)
        i = np.uint32(i * np.uint32(0xD35A2D97)); i ^= i >> np.uint32(15)
    return np.uint32(i ^ np.uint32(0xE6FE3BEB))


def pcg_unit_floats(state0, n):
    """n successive rand_unit_float(&state) values starting from state0 (Random.hpp:20-29)."""
    with np.errstate(over="ignore"):
        a_pow = np.empty(n, np.uint32); a_pow[0] = 1
        if n > 1:
            a_pow[1:] = _A
            a_pow = np.cumprod(a_pow, dtype=np.uint32)
        geo = np.cumsum(np.concatenate([[np.uint32(0)], a_pow[:-1]]).astype(np.uint32), dtype=np.uint32)  # sum_{j<k} A^j
        states = a_pow * np.uint32(state0) + _C * geo  # state before the k-th draw
        v = states
        v = ((v >> ((v >> np.uint32(28)) + np.uint32(4))) ^ v) * np.uint32(277803737)
        out = (v >> np.uint32(22)) ^ v
    return out.astype(np.float32) * f32(2.0 ** -32)


def random_scene(n, light_every=1000, seed=0x04D15A07, emission=20.0):
    """SURVEY.md §8d C3/C4: BVH_test distribution (Application.cpp:107-121) x,z~U(-100,100), y~U(0,100),
    r~U(0.3,20) scaled by (255/n)^(1/3); 8 Lambertian materials albedo~U(0.2,0.9); every `light_every`-th sphere
    uses an emissive material; ambient 0; camera {0,60,300}->{0,0,-1}, focal 50 (Application.cpp:104)."""
    u = pcg_unit_floats(_hash_u32(seed), 5 * n + 24)
    mat_u = u[:24].reshape(8, 3)
    mats = [_mat(albedo=(f32(0.2) + mat_u[i] * f32(0.7))) for i in range(8)]
    mats.append(_mat(albedo=[1, 1, 1], emission=[emission] * 3))
    d = u[24:].reshape(n, 5)
    scale = f32((255.0 / n) ** (1.0 / 3.0)) if n > 255 else f32(1.0)
    r = (f32(0.3) + d[:, 0] * f32(19.7)) * scale
    geo = np.zeros(n, dtype=SPHERE_DTYPE)
    geo["position"][:, 0] = f32(-100) + d[:, 1] * f32(200)
    geo["position"][:, 1] = d[:, 2] * f32(100)
    geo["position"][:, 2] = f32(-100) + d[:, 3] * f32(200)
    geo["radius_sq"] = r * r
    geo["material_ID"] = np.minimum(7, (d[:, 4] * f32(8)).astype(np.int32))
    geo["material_ID"][::light_every] = 8
    return Scene(name=f"random{n}", geometry=geo, material=np.array(mats, dtype=MATERIAL_DTYPE),
                 camera=dict(eye=(0, 60, 300), dir=(0, 0, -1), focal_length=50.0, exposure=1.0),
                 ambient=(0.0, 0.0, 0.0), hdri=None)


def ggx_random_scene(n, light_every=20, seed=0x66780001):
    """random_scene(n) with materials the GGX closure (the reference's `#define BRDF 1` build, DataStreams.hpp:184-219) has something to do
    with: F0 ~ U(0.3, 1) per channel, roughness ~ U(0.05, 1) — and exactly 0 for material 0, the closure's mirror branch (alpha == 0)."""
    sc = random_scene(n, light_every=light_every)
    u = pcg_unit_floats(_hash_u32(seed), 8 * 4).reshape(8, 4)
    for i in range(8):
        sc["material"][i]["F0"] = f32(0.3) + u[i, :3] * f32(0.7)
        sc["material"][i]["roughness"] = f32(0.0) if i == 0 else f32(0.05) + u[i, 3] * f32(0.95)
    sc["name"] = f"ggx_random{n}"
    return sc


def synthetic_hdri(width=64, height=32, seed=0x5EED):
    """Deterministic equirect RGBA32F test texture (the reference loads env.hdr from disk, Application.cpp:225): values in [0.1, 4)."""
    u = pcg_unit_floats(_hash_u32(seed), width * height * 4).reshape(height, width, 4)
    img = f32(0.1) + u * f32(3.9)
    img[..., 3] = 1.0
    return np.ascontiguousarray(img, np.float32)


def bvh_test_scene(n=255, hdri=None):
    """Scenes::BVH_test as the reference lights it (Application.cpp:102-122): n random spheres under an ambient HDRI sky
    (ambient 1,1,1). The reference draws material ids from an EMPTY material list (undefined behaviour, SURVEY §4); here the
    spheres use the 8 Lambertian materials of random_scene and one in 32 is emissive so that light sampling has work to do."""
    sc = random_scene(n, light_every=32)
    sc["name"] = f"bvh_test{n}"
    sc["ambient"] = (1.0, 1.0, 1.0)
    sc["hdri"] = synthetic_hdri() if hdri is None else hdri
    return sc


def sun_hdri(width=2048, height=1024, sun_dir=(0.35, 0.8, -0.48), sun_radius_deg=1.0, sun_radiance=1.0e4):
    """Deterministic equirect RGBA32F sky with a sun: a disk of `sun_radiance` (warm white) of angular radius `sun_radius_deg` around `sun_dir`
    over a dim coloured sky (horizon about 0.3, zenith a deeper blue, ground 0.05). Texel (i, j) is evaluated in the direction the miss
    shader's lookup shows it at (longitude 2 pi ((i + 0.5) / (w - 1) - 0.5), latitude pi (0.5 - (j + 0.5) / (h - 1))), so almost all of the
    energy sits in a few dozen texels: the case a cosine-sampled bounce finds rarely (B2R_FLAG_SKY_LIGHT)."""
    i = (np.arange(width, dtype=np.float64) + 0.5) / max(width - 1, 1)
    j = (np.arange(height, dtype=np.float64) + 0.5) / max(height - 1, 1)
    phi = 2.0 * np.pi * (i - 0.5); lat = np.pi * (0.5 - j)
    dy = np.sin(lat)[:, None] * np.ones((1, width)); r = np.cos(lat)[:, None]
    dx = r * np.cos(phi)[None, :]; dz = r * np.sin(phi)[None, :]
    up = np.clip(dy, 0.0, 1.0)[..., None]
    sky = (1.0 - up) * np.array([0.30, 0.32, 0.36]) + up * np.array([0.06, 0.10, 0.24])
    sky = np.where((dy < 0.0)[..., None], np.array([0.05, 0.045, 0.04]), sky)
    s = np.asarray(sun_dir, np.float64); s = s / np.linalg.norm(s)
    in_sun = dx * s[0] + dy * s[1] + dz * s[2] >= np.cos(np.radians(sun_radius_deg))
    sky = np.where(in_sun[..., None], sun_radiance * np.array([1.0, 0.95, 0.85]), sky)
    img = np.ones((height, width, 4), np.float32); img[..., :3] = sky
    return np.ascontiguousarray(img, np.float32)
