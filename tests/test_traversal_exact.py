"""BVH hit decisions == brute force, exactly, on rays aimed at the mechanisms that make the traversal tree conservative (DESIGN §2):
the per-ray slab set-up (tiny and zero direction components), the leaf cubes sized for the noise of the float sphere tests (rays
bisected to the last ulp the float test still calls a hit), the slab widening (rays through box corners, edges and along faces),
the tie rule and [0, tfar) (duplicate, touching and nested spheres, tfar at a hit distance) and the origin box (origins inside
spheres, far away, non-finite).

CPU tier: every family through every tree kind of tests/hostcheck (the product's own B2R_HD traversal compiled with g++), through
the closest-hit walk k_intersect_closest runs and the any-hit walk k_intersect_shadow runs (TravAnyT), once from the root and once
climbing from each ray's origin sphere as the kernel does, against brute force over all spheres. GPU tier: the
same families through b2r_trace_closest / b2r_trace_shadow for every tree flag, and the frame kernels (BVH vs brute force on the GPU)
on scenes aimed at the same mechanisms. Every comparison is exact: prim ids and tfar bits, occlusion, bucket sums bit for bit."""
import ctypes as C

import numpy as np
import pytest

import b2r
import oracle_py
import scenes

F32_MAX = np.float32(3.4028234663852886e38)
KINDS = {"reference": 0, "sah": 1, "packed": 2, "sweep": 3, "sweep3": 4, "refit": 5}


def _declare(hc):
    vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int
    tree = [i32, vp, vp, u32, vp, u32, vp]
    hc.hc_trace_closest.argtypes = tree + [vp, u32, i32, vp, vp]; hc.hc_trace_closest.restype = i32
    hc.hc_trace_any.argtypes = tree + [vp, vp, vp, u32, vp]; hc.hc_trace_any.restype = i32
    hc.hc_tree_boxes.argtypes = tree + [vp, u32, vp, C.POINTER(u32)]; hc.hc_tree_boxes.restype = i32
    hc.hc_closest_brute.argtypes = [vp, u32, vp, u32, vp, vp]; hc.hc_closest_brute.restype = None
    hc.hc_closest_brute_scalar.argtypes = [vp, u32, vp, u32, vp, vp]; hc.hc_closest_brute_scalar.restype = None
    hc.hc_any_brute.argtypes = [vp, u32, vp, vp, u32, vp]; hc.hc_any_brute.restype = None
    return hc


@pytest.fixture(scope="module")
def hc(hostcheck):
    return _declare(hostcheck)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class Case:
    """One family: spheres (geometry order), rays (n, 6), tfar, the sphere each shadow ray starts from, an origin box or None."""

    def __init__(self, name, geometry, rays, tfar=None, origin_prim=None, box6=None, tail=True):
        self.name = name
        self.geometry = np.ascontiguousarray(geometry, dtype=scenes.SPHERE_DTYPE)
        self.nodes, self.prims, self.ids = b2r.build_bvh(self.geometry)
        self.rays = np.ascontiguousarray(rays, np.float32)
        n = len(self.rays)
        self.tfar = np.ascontiguousarray(np.full(n, 1e30, np.float32) if tfar is None else tfar, np.float32)
        if origin_prim is None:  # in geometry order; the climbing walk starts from any leaf and still searches the whole tree
            origin_prim = np.random.RandomState(n).randint(0, len(self.geometry), n)
        prim_of_geom = np.zeros(len(self.ids), np.int32); prim_of_geom[self.ids] = np.arange(len(self.ids), dtype=np.int32)
        self.origin_prim = np.ascontiguousarray(prim_of_geom[np.asarray(origin_prim)], np.int32)
        self.box6 = None if box6 is None else np.ascontiguousarray(box6, np.float32)
        self.tail = tail  # the scalar tail keeps a NaN distance as its best (BVH.hpp:270-286): compared on finite origins only


def _moved_copy(prims):
    """the spheres a refitted tree was built over: every sphere displaced, same order (HC_REFIT refits the tree to the real ones)"""
    a = prims.copy(); rs = np.random.RandomState(5)
    r = np.sqrt(a["radius_sq"].astype(np.float64))[:, None]
    a["position"] = (a["position"] + rs.uniform(-2, 2, a["position"].shape) * (r + 1.0)).astype(np.float32)
    return a


def host_closest(hc, case, kind, tail=False):
    n = len(case.rays); t = np.empty(n, np.float32); p = np.empty(n, np.int32)
    prims, moved = (_moved_copy(case.prims), case.prims) if kind == KINDS["refit"] else (case.prims, None)
    rc = hc.hc_trace_closest(kind, _p(prims), _p(case.nodes), len(case.nodes), _p(moved), len(case.prims), _p(case.box6), _p(case.rays), n, int(tail), _p(t), _p(p))
    return rc, t, p


def host_any(hc, case, kind, climb=False):
    n = len(case.rays); o = np.empty(n, np.uint8)
    prims, moved = (_moved_copy(case.prims), case.prims) if kind == KINDS["refit"] else (case.prims, None)
    args = (kind, _p(prims), _p(case.nodes), len(case.nodes), _p(moved), len(case.prims), _p(case.box6), _p(case.rays), _p(case.tfar))
    rc = hc.hc_trace_any(*args, _p(case.origin_prim) if climb else None, n, _p(o))
    return rc, o


def brute(hc, case):
    n = len(case.rays)
    t = np.empty(n, np.float32); p = np.empty(n, np.int32); ts = np.empty(n, np.float32); ps = np.empty(n, np.int32); o = np.empty(n, np.uint8)
    hc.hc_closest_brute(_p(case.prims), len(case.prims), _p(case.rays), n, _p(t), _p(p))
    hc.hc_closest_brute_scalar(_p(case.prims), len(case.prims), _p(case.rays), n, _p(ts), _p(ps))
    hc.hc_any_brute(_p(case.prims), len(case.prims), _p(case.rays), _p(case.tfar), n, _p(o))
    return t, p, ts, ps, o


def host_mismatches(hc, case):
    """{(walk, tree kind): number of rays whose result differs from brute force} over every tree kind and walk; only non-zero entries"""
    t0, p0, ts0, ps0, o0 = brute(hc, case)
    finite = np.isfinite(case.rays[:, :3]).all(axis=1)
    bad = {}
    for name, kind in KINDS.items():
        rc, t, p = host_closest(hc, case, kind)
        if rc == 1: continue  # a sweep tree too deep for kTraversalStack: the library builds the packed tree instead
        assert rc == 0, (case.name, name, rc)
        bad[("closest", name)] = int(((p != p0) | (t.view(np.uint32) != t0.view(np.uint32))).sum())
        if case.tail:
            rc, t, p = host_closest(hc, case, kind, tail=True); assert rc == 0
            bad[("closest_tail", name)] = int((((p != ps0) | (t.view(np.uint32) != ts0.view(np.uint32))) & finite).sum())
        rc, o = host_any(hc, case, kind); assert rc == 0
        bad[("any", name)] = int((o != o0).sum())
        rc, o = host_any(hc, case, kind, climb=True); assert rc == 0
        bad[("any_climb", name)] = int((o != o0).sum())
    return {k: v for k, v in bad.items() if v}


def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _rays(o, d):
    r = np.zeros((len(o), 6), np.float32); r[:, :3] = o; r[:, 3:] = d; return r


def _shifted(geo, off):
    g = geo.copy(); g["position"] = (g["position"].astype(np.float64) + off).astype(np.float32); return g


# ------------------------------------------------------------------------------------------------ the families
def family_directions(offset=0.0, lift=400.0, n_spheres=2000):
    """Rays straight down an axis onto random sphere centres, the other two components +-0, subnormal or from a log grid 1e-45..1e-20
    (one and two at a time), in each of the three axis roles. Origins `lift` above the spheres; the scene shifted by `offset`."""
    geo = _shifted(scenes.random_scene(n_spheres, light_every=50)["geometry"], offset)
    rs = np.random.RandomState(int(lift) + int(offset) % 9973)
    eps = np.concatenate([[0.0, -0.0, 1e-45, 1e-42, 1e-40, 3e-39, 1e-38, 5e-38, 1e-37], np.logspace(-45, -20, 14)]).astype(np.float32)
    o, d = [], []
    for main in range(3):
        others = [k for k in range(3) if k != main]
        for e in eps:
            for which in ([others[0]], [others[1]], others):
                c = geo["position"][rs.randint(0, len(geo), 8)].astype(np.float64)
                dd = np.zeros((8, 3), np.float32); dd[:, main] = -1.0
                for k in which: dd[:, k] = e * rs.choice([-1.0, 1.0], 8).astype(np.float32)
                if e == 0.0 and np.signbit(e):
                    for k in which: dd[:, k] = np.float32(-0.0)
                oo = c.copy(); oo[:, main] += lift
                o.append(oo); d.append(dd)
    return Case(f"directions(offset={offset:g}, lift={lift:g})", geo, _rays(np.concatenate(o), np.concatenate(d)))


def _sphere4(s):
    return np.array([s["position"][0], s["position"][1], s["position"][2], s["radius_sq"]], np.float32)


def _last_hit(pred, lo, hi):
    """bisect the offset until lo (hit) and hi (miss) are adjacent floats; returns lo"""
    lo, hi = np.float32(lo), np.float32(hi)
    while np.nextafter(lo, hi) != hi:
        mid = np.float32((np.float64(lo) + np.float64(hi)) / 2)
        if mid == lo or mid == hi: break
        if pred(mid): lo = mid
        else: hi = mid
    return lo


def family_grazing(hc, test, offset=0.0, n_spheres=300, seed=3):
    """For each small sphere (r^2 << 1.5e-6 D^2), a ray from a corner of the origin box (largest D) whose perpendicular offset from the
    centre is bisected over float ulps to the LARGEST offset the float `test` ('closest' FMA, 'tail' scalar, 'any') still calls a hit:
    the rays the leaf cube must contain. box6 = the tight box of spheres and corners, so D is as large as the leaf is sized for."""
    rs = np.random.RandomState(seed)
    geo = np.zeros(n_spheres, scenes.SPHERE_DTYPE)
    geo["position"] = (rs.uniform(-30, 30, (n_spheres, 3)) + offset).astype(np.float32)
    geo["radius_sq"] = (rs.choice([1e-3, 1e-2, 0.05, 0.3], n_spheres) ** 2).astype(np.float32)
    span = np.float64(rs.choice([1e2, 1e3, 1e4]))
    lo = np.float32(offset - span); hi = np.float32(offset + span)
    box6 = np.array([lo, lo, lo, hi, hi, hi], np.float32)
    corners = np.array([[x, y, z] for x in (lo, hi) for y in (lo, hi) for z in (lo, hi)], np.float32)
    rays = []
    for j in range(n_spheres):
        s4 = _sphere4(geo[j]); c = s4[:3].astype(np.float64); r = np.sqrt(np.float64(s4[3]))
        o = corners[rs.randint(8)].astype(np.float64)
        axis = _unit(c - o); u = _unit(np.cross(axis, rs.randn(3)))
        def ray_at(p):
            return np.concatenate([o, _unit(c + np.float64(p) * u - o)]).astype(np.float32)
        def pred(p):
            ray = ray_at(p)
            if test == "closest":
                dd = C.c_float(); return hc.hc_sphere_closest(s4.ctypes.data, ray.ctypes.data, C.byref(dd)) == 1
            if test == "tail":
                b = C.c_float(); pr = C.c_int32(); hc.hc_closest_scalar(s4.ctypes.data, 1, ray.ctypes.data, C.byref(b), C.byref(pr)); return pr.value == 0
            return hc.hc_sphere_any(s4.ctypes.data, ray.ctypes.data, C.c_float(1e30)) == 1
        far = r + 4.0 * np.sqrt(1.5e-6) * np.linalg.norm(c - o)
        if not pred(0.0) or pred(far): continue   # (a tiny sphere far away can be missed by the float ray aimed at its centre)
        rays.append(ray_at(_last_hit(pred, 0.0, far)))
    return Case(f"grazing({test}, offset={offset:g})", geo, np.array(rays), box6=box6)


def family_box_features(hc, kind, n_rays=3000, seed=4):
    """Rays through the corners and edge midpoints of the tree's own slot boxes (entry == exit), and rays that skim a box face: origin
    on the face plane, direction in the plane or tilted out of it by a few ulps. A box rejected by rounding shows as a lost hit."""
    rs = np.random.RandomState(seed + kind)
    sc = scenes.random_scene(1500, light_every=50)
    # one explicit origin box for the tree the boxes are read from and the tree the rays are traced through (the leaf extents depend on it)
    box6 = FEATURE_BOX
    case = Case("features", sc["geometry"], np.zeros((1, 6), np.float32), box6=box6)
    prims, moved = (_moved_copy(case.prims), case.prims) if kind == KINDS["refit"] else (case.prims, None)
    m = C.c_uint32(0)
    args = (kind, _p(prims), _p(case.nodes), len(case.nodes), _p(moved), len(case.prims), _p(case.box6), None, 0)
    assert hc.hc_tree_boxes(*args, None, C.byref(m)) in (0, 1)
    boxes = np.zeros((m.value, 7), np.float32)
    if hc.hc_tree_boxes(*args, _p(boxes), C.byref(m)) == 1: return None
    rays = feature_rays(boxes[:, 0:3], boxes[:, 3:6], box6[:3], box6[3:], n_rays, rs)
    return Case(f"box features (tree {kind})", sc["geometry"], rays, box6=box6)


# origin box of family 3 on the CPU: holds the random_scene spheres (x, z in -111..111, y in -11..111) and the ray origins
FEATURE_BOX = np.array([-160, -60, -160, 160, 160, 160], np.float32)


def feature_rays(box_lo, box_hi, o_lo, o_hi, n_rays, rs):
    """rays through the corners and edge midpoints of the given slot boxes and along their faces; origins inside [o_lo, o_hi] (the origin
    box the tree was sized for, shrunk by 1 %, so that tracing them does not grow it)"""
    o_lo = np.asarray(o_lo, np.float64); o_hi = np.asarray(o_hi, np.float64)
    o_lo, o_hi = o_lo + 0.01 * (o_hi - o_lo), o_hi - 0.01 * (o_hi - o_lo)
    idx = rs.randint(0, len(box_lo), n_rays)
    lo, hi = box_lo[idx].astype(np.float64), box_hi[idx].astype(np.float64)
    sel = rs.randint(0, 2, (n_rays, 3)).astype(bool)
    target = np.where(sel, lo, hi)
    kindsel = rs.randint(0, 3, n_rays)   # 0: corner, 1: edge midpoint, 2: along a face
    edge_axis = rs.randint(0, 3, n_rays)
    mid = 0.5 * (lo + hi)
    target[kindsel == 1, edge_axis[kindsel == 1]] = mid[kindsel == 1, edge_axis[kindsel == 1]]
    o = rs.uniform(o_lo, o_hi, (n_rays, 3))
    d = _unit(target - o)
    face = kindsel == 2
    fa = edge_axis[face]
    o_face = o[face]; o_face[np.arange(face.sum()), fa] = target[face, fa]       # origin in the face plane ...
    d_face = _unit(rs.randn(face.sum(), 3)); d_face[np.arange(face.sum()), fa] = 0.0  # ... direction in it
    tilt = rs.choice([0.0, 1e-7, -1e-7, 1e-30], face.sum()); d_face[np.arange(face.sum()), fa] = tilt
    o[face] = o_face; d[face] = d_face
    o = np.clip(o, o_lo, o_hi)
    rays = _rays(o.astype(np.float32), d.astype(np.float32))
    return rays[np.abs(rays[:, 3:]).max(axis=1) > 0]


def family_ties(n_rays=2000, seed=6):
    """Coincident duplicates (the lowest index wins, BVH.hpp:265), touching pairs, nested (concentric and off-centre) spheres; closest
    rays through contact points, shadow rays leaving a sphere's surface toward another, and tfar exactly at the brute-force hit distance
    (the interval is [0, tfar): the sphere at distance tfar does not occlude) and one ulp above it."""
    rs = np.random.RandomState(seed)
    base = np.zeros(60, scenes.SPHERE_DTYPE)
    base["position"] = rs.uniform(-20, 20, (60, 3)).astype(np.float32); base["radius_sq"] = (rs.uniform(0.5, 3, 60) ** 2).astype(np.float32)
    dup = base[rs.randint(0, 60, 30)]                                    # coincident duplicates
    touch = base[:30].copy(); r0 = np.sqrt(base["radius_sq"][:30].astype(np.float64)); r1 = rs.uniform(0.5, 2, 30)
    dirs = _unit(rs.randn(30, 3)); touch["position"] = (base["position"][:30] + dirs * (r0 + r1)[:, None]).astype(np.float32)
    touch["radius_sq"] = (r1 ** 2).astype(np.float32)
    nest = base[30:].copy(); nest["radius_sq"] = (base["radius_sq"][30:] * 0.25).astype(np.float32)       # concentric
    nest2 = base[30:].copy(); nest2["position"] = (base["position"][30:] + 0.3 * dirs).astype(np.float32); nest2["radius_sq"] = (base["radius_sq"][30:] * 0.5).astype(np.float32)
    geo = np.concatenate([base, dup, touch, nest, nest2])
    pos = geo["position"].astype(np.float64); rad = np.sqrt(geo["radius_sq"].astype(np.float64))
    contact = base["position"][:30].astype(np.float64) + dirs * r0[:, None]
    o, d, origin = [], [], []
    for i in range(n_rays):
        k = rs.randint(4)
        if k == 0:    # at a contact point or a duplicated sphere from outside
            tgt = contact[rs.randint(30)] if rs.rand() < 0.5 else pos[60 + rs.randint(30)]
            oo = tgt + _unit(rs.randn(3)) * 60; origin.append(rs.randint(len(geo)))
        else:         # from a sphere's surface (the shading offset of 1e-4 along the normal, or none), toward another sphere
            s = rs.randint(len(geo)); nrm = _unit(rs.randn(3))
            oo = pos[s] + nrm * (rad[s] + (1e-4 if k == 1 else 0.0)); tgt = pos[rs.randint(len(geo))] + rs.randn(3) * 0.5
            origin.append(s)
        o.append(oo); d.append(_unit(tgt - oo))
    return geo, _rays(np.array(o, np.float32), np.array(d, np.float32)), np.array(origin)


def ties_case(hc):
    geo, rays, origin = family_ties()
    probe = Case("ties", geo, rays, origin_prim=origin)
    t, p, _, _, _ = brute(hc, probe)
    hit = p >= 0
    tfar = np.where(hit, t, np.float32(50.0)).astype(np.float32)
    sel = np.random.RandomState(8).randint(0, 3, len(rays))
    tfar = np.where(sel == 1, np.nextafter(tfar, F32_MAX), tfar)                 # one ulp above the hit
    tfar = np.where(sel == 2, np.float32(1e30), tfar).astype(np.float32)         # unbounded
    return Case("ties", geo, rays, tfar=tfar, origin_prim=origin)


def family_origins(seed=9):
    """Origins inside spheres, far outside the sphere bounds (1e3..1e15 away, inside the claim's 2^61) and non-finite (inf, -inf, NaN in
    one component or all), aimed at random spheres. The origin box is grown over the finite origins only, as b2r_trace_* does."""
    rs = np.random.RandomState(seed)
    geo = scenes.random_scene(1200, light_every=40)["geometry"]
    pos = geo["position"].astype(np.float64); rad = np.sqrt(geo["radius_sq"].astype(np.float64))
    o, d = [], []
    for i in range(1500):
        s = rs.randint(len(geo)); k = rs.randint(3)
        if k == 0: oo = pos[s] + _unit(rs.randn(3)) * rad[s] * rs.uniform(0, 0.99)
        elif k == 1: oo = pos[s] + _unit(rs.randn(3)) * 10.0 ** rs.uniform(3, 15)
        else: oo = pos[s] + _unit(rs.randn(3)) * 500
        o.append(oo); d.append(_unit(pos[rs.randint(len(geo))] + rs.randn(3) - oo) if k != 1 else _unit(pos[s] + rs.randn(3) * rad[s] - oo))
    o = np.array(o, np.float32); d = np.array(d, np.float32)
    nf = rs.choice(len(o), 300, replace=False)
    for j, i in enumerate(nf):
        v = [np.inf, -np.inf, np.nan][j % 3]
        if j % 2: o[i, j % 3] = v
        else: o[i, :] = v
    return Case("origins", geo, _rays(o, d), tfar=rs.uniform(1, 1e4, len(o)).astype(np.float32))


def family_stack_quantum(n_rays=10000, seed=1):
    """C3's 100k spheres under C3's camera. With ~35k wide nodes a traversal stack entry keeps 16 bits of its entry distance (8 mantissa
    bits, a quantum of 2^-8 relative), so a popped node is often entered within one quantum of the best distance found so far: the entry
    must be a lower bound (pack_entry truncates) or the node holding a slightly nearer hit is culled."""
    rs = np.random.RandomState(seed)
    o = np.tile(np.array([0.0, 60.0, 300.0]), (n_rays, 1))
    d = _unit(np.c_[rs.uniform(-0.35, 0.35, n_rays), rs.uniform(-0.35, 0.15, n_rays), -np.ones(n_rays)])
    return Case("stack quantum", scenes.random_scene(100000)["geometry"], _rays(o, d), tail=False)


def _assert_exact(bad, case):
    assert not bad, f"{case.name}: rays differing from brute force per (walk, tree): {bad}"


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("offset,lift", [(0.0, 400.0), (0.0, 3e4), (1e4, 400.0), (1e6, 2e5)])
def test_tiny_direction_components_equal_brute_force(hc, offset, lift):
    """Family 1: +-0, subnormal and tiny direction components. A finite 1/d with |o/d| > FLT_MAX must not reject boxes (slab_setup)."""
    case = family_directions(offset, lift)
    t0, p0, _, _, _ = brute(hc, case)
    assert (p0 >= 0).mean() > 0.9   # the rays are aimed at sphere centres: brute force hits almost all of them
    _assert_exact(host_mismatches(hc, case), case)


@pytest.mark.parametrize("test", ["closest", "tail", "any"])
@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_grazing_rays_at_the_noise_bound(hc, test, offset):
    """Family 2: the last float ulp of perpendicular offset each sphere test still calls a hit, from the origin box's corners."""
    case = family_grazing(hc, test, offset)
    assert len(case.rays) > 100, len(case.rays)
    _assert_exact(host_mismatches(hc, case), case)


@pytest.mark.parametrize("kind", list(KINDS.values()))
def test_rays_through_box_corners_edges_and_faces(hc, kind):
    """Family 3: rays whose entry and exit coincide on the slot boxes of the tree under test (the slab widening's case)."""
    case = family_box_features(hc, kind)
    if case is None: pytest.skip("sweep tree too deep for this scene (the library builds the packed tree instead)")
    _assert_exact(host_mismatches(hc, case), case)


def test_ties_contact_and_tfar_boundaries(hc):
    """Family 4: equal distances go to the lowest index in every walk; shadow rays from sphere surfaces; tfar exactly at a hit."""
    case = ties_case(hc)
    t0, p0, _, _, o0 = brute(hc, case)
    assert (p0 >= 0).mean() > 0.5 and 0.1 < o0.mean() < 0.95
    _assert_exact(host_mismatches(hc, case), case)


def test_origins_inside_far_and_non_finite(hc):
    """Family 5: origins inside spheres, 1e3..1e15 away, and non-finite (the walk then tests every sphere, as brute force does)."""
    case = family_origins()
    _assert_exact(host_mismatches(hc, case), case)


def test_stack_entry_distance_is_a_lower_bound_at_100k_spheres(hc):
    """Closest hits at C3's size, where the stack entries are coarsest: every tree kind equals brute force exactly."""
    case = family_stack_quantum()
    t0, p0, _, _, _ = brute(hc, case)
    assert (p0 >= 0).mean() > 0.5
    bad = {}
    for name, kind in KINDS.items():
        rc, t, p = host_closest(hc, case, kind)
        if rc == 1: continue
        assert rc == 0, (name, rc)
        bad[("closest", name)] = int(((p != p0) | (t.view(np.uint32) != t0.view(np.uint32))).sum())
    _assert_exact({k: v for k, v in bad.items() if v}, case)


# ------------------------------------------------------------------------------------------------ GPU tier
TREE_FLAGS = {"default": 0, "reference": b2r.FLAG_REFERENCE_TREE, "gpu_packed": b2r.FLAG_GPU_TREE,
              "gpu_sweep": b2r.FLAG_GPU_TREE | b2r.FLAG_GPU_SAH, "gpu_sweep3": b2r.FLAG_GPU_TREE | b2r.FLAG_GPU_SAH3}


def _scene_of(geometry):
    sc = scenes.random_scene(len(geometry), light_every=40)
    sc["geometry"] = np.ascontiguousarray(geometry, dtype=scenes.SPHERE_DTYPE)
    sc["geometry"]["material_ID"] = np.where(np.arange(len(geometry)) % 40 == 0, 8, np.arange(len(geometry)) % 8)
    return sc


def _gpu_cases(hc):
    return [family_directions(0.0, 400.0), family_directions(1e4, 400.0), family_directions(1e6, 2e5), family_grazing(hc, "closest"),
            family_grazing(hc, "any", 1e4), ties_case(hc), family_origins()]


def _gpu_feature_case(r, geometry, seed=4):
    """family 3 on the device: rays through the corners, edges and faces of the slot boxes the renderer traces right now (its own tree, leaf
    extents sized for its current origin box), with origins inside that box so that tracing them leaves the tree as it is"""
    wide, _ = r.wide_nodes(); box = r.origin_box()
    used = wide[:, :, 6].view(np.int32) != np.int32(-2 ** 31)
    c, h = wide[:, :, 0:3][used], wide[:, :, [4, 5, 7]][used]
    rays = feature_rays(c - h, c + h, box[:3], box[3:], 3000, np.random.RandomState(seed))
    return Case("box features (device tree)", geometry, rays)


def _gpu_trace_matches_oracle(r, o, case):
    t, p = r.trace_closest(case.rays); to, po = o.trace_closest(case.rays)
    occ = r.trace_shadow(case.rays, case.tfar); occ_o = o.trace_shadow(case.rays, case.tfar)
    bad = {"closest": int(((p != po) | (t.view(np.uint32) != to.view(np.uint32))).sum()), "any": int((occ != occ_o).sum())}
    return {k: v for k, v in bad.items() if v}


@pytest.mark.gpu
@pytest.mark.parametrize("tree", list(TREE_FLAGS) + ["refit"])
def test_gpu_trace_api_exact_on_adversarial_families(hc, tree):
    """b2r_trace_closest / b2r_trace_shadow (k_tap_trace) on every family, for every tree flag and after a RefitScene, against the
    oracle's brute force, exactly; family 3 is aimed at the boxes of the device tree itself. Then a batch from far outside the origin box
    (the box grows and the device tree is refitted) and the families again."""
    fails = []
    flags = b2r.FLAG_FORCE_BVH | TREE_FLAGS.get(tree, 0)
    def renderer(sc):
        if tree != "refit": return b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=flags)
        sa = scenes.Scene(sc); sa["geometry"] = _moved_copy(sc["geometry"])   # built over displaced spheres, then refitted to the real ones
        r = b2r.Renderer(sa, 64, 64, max_bounces=4, buckets=1, flags=flags); r.RefitScene(sc["geometry"])
        return r
    sc = _scene_of(scenes.random_scene(1500, light_every=50)["geometry"])   # family 3 on the tree under test
    r = renderer(sc); o = oracle_py.Oracle(64, 64, max_bounces=4, K=1); o.set_scene(sc)
    box = r.origin_box(); case = _gpu_feature_case(r, sc["geometry"])
    bad = _gpu_trace_matches_oracle(r, o, case)
    assert np.array_equal(r.origin_box(), box)   # traced through exactly the boxes the rays were aimed at
    if bad: fails.append((case.name, "", bad))
    r.close(); o.close()
    for case in _gpu_cases(hc):
        sc = _scene_of(case.geometry)
        r = renderer(sc)
        o = oracle_py.Oracle(64, 64, max_bounces=4, K=1); o.set_scene(sc)
        bad = _gpu_trace_matches_oracle(r, o, case)
        if bad: fails.append((case.name, "", bad))
        box = r.origin_box()
        far = case.rays[np.isfinite(case.rays[:, :3]).all(axis=1)][:512].copy()
        far[:, :3] += np.float32(4.0) * (box[3:] - box[:3])           # origins far outside the current origin box
        fcase = Case(case.name + " far", case.geometry, far, tail=False)
        bad = _gpu_trace_matches_oracle(r, o, fcase)
        assert not np.array_equal(r.origin_box(), box)
        if bad: fails.append((case.name, "far batch", bad))
        bad = _gpu_trace_matches_oracle(r, o, case)                   # and the families again, inside the grown box
        if bad: fails.append((case.name, "after growth", bad))
        r.close(); o.close()
    assert not fails, f"tree {tree}: {fails}"


def _frame_scenes():
    shifted = scenes.random_scene(3000, light_every=40)
    shifted["geometry"] = _shifted(shifted["geometry"], 1e4)
    shifted["camera"] = dict(eye=(1e4, 1e4 + 60, 1e4 + 300), dir=(0, 0, -1), focal_length=50.0, exposure=1.0)
    tiny = scenes.random_scene(4000, light_every=20)
    tiny["geometry"]["radius_sq"] = (tiny["geometry"]["radius_sq"] * np.float32(1e-4)).astype(np.float32)
    tiny["geometry"]["radius_sq"][::20] = np.float32(400.0)
    tiny["camera"] = dict(eye=(0, 50, 4e4), dir=(0, 0, -1), focal_length=8000.0, exposure=1.0)
    geo, _, _ = family_ties()
    ties = _scene_of(geo)
    ties["camera"] = dict(eye=(0, 0, 70), dir=(0, 0, -1), focal_length=30.0, exposure=1.0)
    big = scenes.random_scene(300000, light_every=300)   # > 65 536 wide nodes: the stack-entry split is read from the scene
    return {"shifted_1e4": shifted, "tiny_far_camera": tiny, "ties": ties, "over_65536_nodes": big}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["shifted_1e4", "tiny_far_camera", "ties", "over_65536_nodes"])
@pytest.mark.parametrize("no_packet", [False, True])
def test_gpu_frame_bvh_equals_brute_bit_for_bit(name, no_packet, monkeypatch):
    """k_intersect_packet (or, with B2R_NO_PACKET=1, the staged k_intersect_closest at bounce 0), k_intersect_closest and the climbing
    k_intersect_shadow against the brute-force kernels on the GPU: bucket sums bit-identical."""
    if no_packet: monkeypatch.setenv("B2R_NO_PACKET", "1")
    else: monkeypatch.delenv("B2R_NO_PACKET", raising=False)
    sc = _frame_scenes()[name]
    w, h = (320, 192) if name != "over_65536_nodes" else (640, 384)
    ps = b2r.PreparedScene(sc, w, h)
    a = b2r.Renderer(ps, w, h, max_bounces=8, buckets=1, flags=b2r.FLAG_FORCE_BVH); a.Accumulate(2)
    b = b2r.Renderer(ps, w, h, max_bounces=8, buckets=1, flags=b2r.FLAG_FORCE_BRUTE); b.Accumulate(2)
    ga, gb = a.buckets_host(), b.buckets_host()
    if name == "over_65536_nodes": assert len(a.wide_nodes()[0]) > 65536
    ca, cb = a.counters(), b.counters()
    print(f"{name} no_packet={no_packet}: bit-identical {ga.tobytes() == gb.tobytes()}, rays {ca['extension_rays']} / {cb['extension_rays']}, shadow rays {ca['shadow_rays']}")
    assert float(ga.max()) > 0.0 and ca["shadow_rays"] > 0
    assert ga.tobytes() == gb.tobytes()
    assert ca["extension_rays"] == cb["extension_rays"]
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("tree", ["default", "gpu_sweep3"])
def test_gpu_camera_leaving_the_origin_box_back_to_back(tree):
    """The camera jumps far outside the origin box between frames enqueued back to back (RenderDevice, no host wait): the box grows and
    the tree is refitted on the device, and the frame must trace the refitted tree. A pipelined renderer runs every prefix of the camera
    path, so that each far jump is the LAST frame of one run, where it is read: it must equal the same frame of a renderer that waits
    after every call, and brute force."""
    sc = scenes.random_scene(5000, light_every=40)
    w, h, K = 192, 128, 2
    ps = b2r.PreparedScene(sc, w, h)
    eyes = [(0, 60, 300), (0, 60, 3e4), (2e4, 5e3, -2e4), (0, 60, 300), (-9e4, 2e4, 1e3)]
    grows = [False, True, True, False, True]   # whether the eye lies outside the box grown by the eyes before it
    look = np.array([0, 30, 0], np.float64)   # the focal length grows with the distance, so that every frame sees the scene at about the same size
    cams = [b2r.camera_lookat(e, _unit(look - np.array(e)), w, h, 50.0 * max(1.0, float(np.linalg.norm(look - np.array(e))) / 300.0), 1.0) for e in eyes]
    flags = b2r.FLAG_FORCE_BVH | TREE_FLAGS[tree]
    def run(r, cams, wait):
        out, boxes = [], []
        for cam in cams:
            boxes.append(r.origin_box())
            r.SetCamera(cam); r.ResetAccumulator(); r.Accumulate(K)
            assert r.RenderDevice()
            if wait: r.sync(); out.append(r.buckets_host())
        boxes.append(r.origin_box())
        if not wait: r.sync(); out.append(r.buckets_host())
        return out, boxes
    waited = b2r.Renderer(ps, w, h, max_bounces=8, buckets=K, flags=flags); ref, boxes = run(waited, cams, True)
    brute_r = b2r.Renderer(ps, w, h, max_bounces=8, buckets=K, flags=b2r.FLAG_FORCE_BRUTE); ref_b, _ = run(brute_r, cams, True)
    assert [not np.array_equal(boxes[i], boxes[i + 1]) for i in range(len(eyes))] == grows
    for i in range(len(eyes)):
        assert ref[i].tobytes() == ref_b[i].tobytes(), f"frame {i} (eye {eyes[i]}): BVH differs from brute force"
        assert float(ref[i].max()) > 0.0
    for n in range(2, len(eyes) + 1):
        piped = b2r.Renderer(ps, w, h, max_bounces=8, buckets=K, flags=flags)
        got, pboxes = run(piped, cams[:n], False)
        assert np.array_equal(pboxes[-1], boxes[n])
        assert got[-1].tobytes() == ref[n - 1].tobytes(), f"pipelined run ending on eye {eyes[n - 1]} (growth: {grows[n - 1]}) differs"
        piped.close()
    waited.close(); brute_r.close()
