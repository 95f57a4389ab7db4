"""The traversal kernels a frame is traced with, on the adversarial ray families of tests/test_traversal_exact.py, against brute force,
exactly (prim ids, tfar bits, occlusion). b2r_trace_closest / b2r_trace_shadow run k_tap_trace, a root walk with its own stack; every
frame is traced by three other kernels, reached here through b2r_trace_kernel with the instantiation and grid a frame would use:
k_intersect_closest (nodes staged through shared memory, the 16-entry shared stack that spills to local memory, the stack-entry split as an
immediate up to 65 536 wide nodes and read from the scene above, lane refill, the scalar tail of B2R_FLAG_REFERENCE_EXACT),
k_intersect_shadow (the walk from the origin sphere's leaf, climbing through parent[]) and k_intersect_packet (one walk per warp for the
camera rays). Also: the link tables k_link_tables writes (parent[] and leaf_node[], where the shadow walks start and how they climb)
against the tree's own links, the refit quality ratio against a float64 host sum, and that the taps leave a renderer's frames alone.

CPU tier: the error returns that need no device and the set-up of the tiny-component cameras. GPU tier: everything else (-m gpu)."""
import ctypes as C

import numpy as np
import pytest

import b2r
import scenes
from conftest import have_gpu
from test_traversal_exact import (TREE_FLAGS, Case, _declare, _gpu_cases, _gpu_feature_case, _last_hit, _moved_copy, _rays, _scene_of,
                                  _shifted, _unit, family_grazing, family_ties, family_stack_quantum)

INT32_MIN = np.int32(-2 ** 31)   # kEmptyLink
needs_gpu = pytest.mark.skipif(not have_gpu(), reason="needs a CUDA device")


@pytest.fixture(scope="module")
def hc(hostcheck):
    return _declare(hostcheck)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def brute_closest(hc, prims, rays, scalar=False):
    n = len(rays); t = np.empty(n, np.float32); p = np.empty(n, np.int32)
    (hc.hc_closest_brute_scalar if scalar else hc.hc_closest_brute)(_p(prims), len(prims), _p(rays), n, _p(t), _p(p))
    return t, p


def brute_any(hc, prims, rays, tfar):
    n = len(rays); o = np.empty(n, np.uint8)
    hc.hc_any_brute(_p(prims), len(prims), _p(rays), _p(tfar), n, _p(o))
    return o


def differ(t, p, t0, p0):
    return (p != p0) | (t.view(np.uint32) != t0.view(np.uint32))


def closest_mismatches(hc, r, rays):
    """rays where the per-lane kernel, and where b2r_trace_closest, differ from brute force over the renderer's BVH-order spheres"""
    prims = np.ascontiguousarray(r.scene.prims); rays = np.ascontiguousarray(rays, np.float32)
    t0, p0 = brute_closest(hc, prims, rays)
    t, p = r.trace_kernel_closest(rays); ta, pa = r.trace_closest(rays)
    return {"closest kernel": int(differ(t, p, t0, p0).sum()), "trace api": int(differ(ta, pa, t0, p0).sum())}


def shadow_batch(case, r):
    """the family's rays three times over and more: from the spheres the family gives (ties: the spheres the rays leave), from the root
    (-1), and in copies whose walks between them start at every sphere of the renderer's BVH order"""
    n, m = len(case.rays), len(r.scene.prims)
    pog = np.empty(m, np.int32); pog[r.scene.prim_ids] = np.arange(m, dtype=np.int32)
    own = pog[case.ids[case.origin_prim]]
    k = -(-m // n)
    cover = np.random.RandomState(m).permutation(np.arange(k * n) % m)
    origin = np.concatenate([own, np.full(n, -1), cover]).astype(np.int32)
    assert set(origin[origin >= 0].tolist()) == set(range(m))
    return np.tile(case.rays, (k + 2, 1)), np.tile(case.tfar, k + 2), origin


def shadow_mismatches(hc, r, case):
    rays, tfar, origin = shadow_batch(case, r)
    o0 = brute_any(hc, np.ascontiguousarray(r.scene.prims), rays, tfar)
    o = r.trace_kernel_shadow(rays, tfar, origin)
    return {"shadow kernel": int((o != o0).sum())}


def _nonzero(bad):
    return {k: v for k, v in bad.items() if v}


def host_link_tables(wide, n_prims):
    """parent[] / leaf_node[] read off the node array: a slot linking inner node l makes its node l's parent, a leaf slot ~l holds sphere l"""
    link = wide[:, :, 6].view(np.int32)
    node = np.repeat(np.arange(len(wide), dtype=np.uint32), 4).reshape(len(wide), 4)
    parent = np.zeros(len(wide), np.uint32); leaf = np.full(n_prims, 0xffffffff, np.uint32)
    inner, lf = link >= 0, (link < 0) & (link != INT32_MIN)
    parent[link[inner]] = node[inner]; leaf[~link[lf]] = node[lf]
    assert (leaf != 0xffffffff).all() and inner.sum() == len(wide) - 1
    return parent, leaf


def assert_link_tables(r, what):
    wide, _ = r.wide_nodes()
    hp, hl = host_link_tables(wide, len(r.scene.prims))
    dp, dl = r.link_tables()
    assert np.array_equal(dp, hp), f"{what}: parent[] differs at {np.flatnonzero(dp != hp)[:10]}"
    assert np.array_equal(dl, hl), f"{what}: leaf_node[] differs at {np.flatnonzero(dl != hl)[:10]}"


def half_area_sum(wide):
    """sum of slot_half_area over the inner slots, each term in float32 as the device forms it, summed in float64"""
    link = wide[:, :, 6].view(np.int32); inner = link >= 0
    hx, hy, hz = wide[:, :, 4][inner], wide[:, :, 5][inner], wide[:, :, 7][inner]
    return (np.float32(4.0) * ((hx * hy + hy * hz) + hz * hx)).astype(np.float64).sum()


def _renderer(sc, tree, w=64, h=64, extra=0, **kw):
    """a BVH renderer with the tree of TREE_FLAGS[tree]; 'refit' / 'refit_keep': built over displaced spheres, then refitted to the real
    ones into a new BVH order (leaves re-linked) / the order it was built with"""
    flags = b2r.FLAG_FORCE_BVH | TREE_FLAGS.get(tree, 0) | extra
    if not tree.startswith("refit"):
        return b2r.Renderer(sc, w, h, max_bounces=4, buckets=1, flags=flags, **kw)
    sa = scenes.Scene(sc); sa["geometry"] = _moved_copy(sc["geometry"])
    r = b2r.Renderer(sa, w, h, max_bounces=4, buckets=1, flags=flags, **kw)
    r.RefitScene(sc["geometry"], keep_order=tree == "refit_keep")
    return r


# ------------------------------------------------------------------------------------------------ CPU tier
def test_trace_kernel_rejects_a_null_context():
    L = b2r.lib()
    assert L.b2r_trace_kernel(None, b2r.TAP_CLOSEST, None, None, None, None, 1, 0, None, None, None) == b2r.ERR_ARG
    assert L.b2r_read_link_tables(None, None, None) == b2r.ERR_ARG


def _tiny_camera(far):
    """camera looking exactly down -z (identity orientation: the x and y components are the pixel offsets scaled by 1/|z|) with |z| =
    1.2e19 in a 16x16 frame, about the largest that keeps |d|^2 finite in float: every x and y component is below 2^-60. far: the eye 1e18 from the origin (inside
    the 2^61 bound), where a kept axis's |o/d| is largest"""
    eye = (1e18, -1e18, 1e18) if far else (0.5, -0.25, 500.0)
    return dict(eye=eye, dir=(0, 0, -1), focal_length=1.8e19, exposure=1.0)   # |z| = (h / 2) * focal / 12


@pytest.mark.parametrize("far", [False, True])
def test_tiny_component_cameras_give_components_below_2_to_minus_60(far):
    """The packet scenes below need camera rays whose x and y components lie below 2^-60, around the 2^-62 where slab_setup stops
    keeping an axis: b2r_camera_ray (the kernels' camera_dir on the host) at the frame's corners and centre."""
    cam = _tiny_camera(far); w = h = 16
    out = b2r.camera_lookat(cam["eye"], cam["dir"], w, h, cam["focal_length"])
    assert tuple(out[3:7]) == (1.0, 0.0, 0.0, 0.0)
    comps = []
    for x, y, s in [(0, 0, 0.0), (15, 15, 0.9999999), (0, 15, 0.5), (8, 8, 0.001), (7, 7, 0.999)]:
        o = np.zeros(3, np.float32); d = np.zeros(3, np.float32); smp = np.array([s, s], np.float32)
        assert b2r.lib().b2r_camera_ray(_p(out[0:3]), _p(out[3:7]), float(out[7]), float(out[8]), float(out[9]), x, y, _p(smp), _p(o), _p(d)) == 0
        assert d[2] == -1.0 and np.isfinite(d).all()
        comps += [abs(float(d[0])), abs(float(d[1]))]
    assert max(comps) < 2.0 ** -60 and max(comps) > 2.0 ** -62 and min(comps) < 1e-20


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.fixture(scope="module")
def families(hc):
    return _gpu_cases(hc)


@pytest.fixture(scope="module")
def c3():
    """C3's 100k spheres (about 35k wide nodes: the stack-entry split is the immediate 16/16)"""
    r = b2r.Renderer(scenes.random_scene(100000), 128, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    yield r
    r.close()


@pytest.fixture(scope="module")
def big():
    """300k spheres: more than 65 536 wide nodes, the split is read from the scene"""
    r = b2r.Renderer(scenes.random_scene(300000, light_every=300), 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    yield r
    r.close()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("tree", list(TREE_FLAGS) + ["refit", "refit_keep"])
def test_gpu_closest_and_shadow_kernels_exact_on_adversarial_families(hc, families, tree):
    """Every family through k_intersect_closest and the climbing k_intersect_shadow, for every tree flag and after a refit into a new
    BVH order (k_link_tables runs again) and into the same one; family 3 aims at the device tree's own slot boxes. The trace API must
    agree as well. Shadow walks start at every sphere, at the root, and at the spheres the ties family's rays really leave."""
    fails = []
    sc = _scene_of(scenes.random_scene(1500, light_every=50)["geometry"])
    r = _renderer(sc, tree)
    case = _gpu_feature_case(r, sc["geometry"]); box = r.origin_box()
    bad = _nonzero({**closest_mismatches(hc, r, case.rays), **shadow_mismatches(hc, r, case)})
    assert np.array_equal(r.origin_box(), box)   # traced through exactly the boxes the rays were aimed at
    if bad: fails.append((case.name, bad))
    r.close()
    for case in families:
        r = _renderer(_scene_of(case.geometry), tree)
        bad = _nonzero({**closest_mismatches(hc, r, case.rays), **shadow_mismatches(hc, r, case)})
        if bad: fails.append((case.name, bad))
        r.close()
    assert not fails, f"tree {tree}: {fails}"


def _nest_scene():
    """the nested spheres of test_deep_traversal_stack_nested_spheres: every box overlaps every other, the per-lane stack grows by three per
    level and its shared part (16 entries) spills on almost every ray"""
    sc = scenes.random_scene(4096, light_every=64)
    rs = np.random.RandomState(7); g = sc["geometry"]
    g["position"][:] = rs.uniform(-1.0, 1.0, (len(g), 3)).astype(np.float32)
    g["radius_sq"][:] = (rs.uniform(5.0, 6.0, len(g)).astype(np.float32)) ** 2
    lights = np.arange(0, len(g), 64); d = _unit(rs.randn(len(lights), 3))
    g["position"][lights] = (40.0 * d).astype(np.float32); g["radius_sq"][lights] = np.float32(4.0)
    return sc


def _nest_case(sc, n=4000, seed=11):
    """rays through the nest: from a shell of radius 30 toward points of the cluster, and from inside the cluster outward"""
    rs = np.random.RandomState(seed)
    o = 30.0 * _unit(rs.randn(n, 3)); o[n // 2:] = rs.uniform(-1, 1, (n - n // 2, 3))
    d = _unit(rs.uniform(-1, 1, (n, 3)) - o); d[n // 2:] = _unit(rs.randn(n - n // 2, 3))
    return Case("nest", sc["geometry"], _rays(o.astype(np.float32), d.astype(np.float32)), tfar=rs.uniform(1, 60, n).astype(np.float32))


@pytest.mark.gpu
@needs_gpu
def test_gpu_closest_kernel_deep_stack_and_count_instantiation(hc, families):
    """The stack_evict / refill() path of the shared-memory stack (nested spheres, rays through the nest) in both kernels that have it, and
    the B2R_FLAG_COUNT_TESTS instantiations of all three kernels, which are separate template instances."""
    sc = _nest_scene()
    r = b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    _, max_stack = r.wide_nodes()
    assert max_stack > 13, max_stack
    case = _nest_case(sc)
    bad = {}
    for flags in (b2r.FLAG_FORCE_BVH, b2r.FLAG_FORCE_BVH | b2r.FLAG_COUNT_TESTS):
        r.set_flags(flags)
        for k, v in {**closest_mismatches(hc, r, case.rays), **shadow_mismatches(hc, r, case)}.items(): bad[(flags, "nest", k)] = v
        t0, p0 = brute_closest(hc, np.ascontiguousarray(r.scene.prims), r.generate_rays(1))
        t, p = r.trace_kernel_packet(1); bad[(flags, "nest", "packet")] = int(differ(t, p, t0, p0).sum())
    r.close()
    dirs = families[0]   # tiny direction components, under the counting instantiation
    r = b2r.Renderer(_scene_of(dirs.geometry), 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | b2r.FLAG_COUNT_TESTS)
    for k, v in {**closest_mismatches(hc, r, dirs.rays), **shadow_mismatches(hc, r, dirs)}.items(): bad[("count", dirs.name, k)] = v
    r.close()
    assert not _nonzero(bad), _nonzero(bad)


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("size", ["c3_100k", "over_65536_nodes"])
def test_gpu_kernels_on_both_sides_of_the_stack_entry_split(hc, c3, big, size):
    """Closest hits where a stack entry keeps only 8 mantissa bits of its distance (family_stack_quantum's rays), through the instantiation
    with the 16/16 split as an immediate (C3, <= 65 536 wide nodes) and the one that reads the split from the scene (300k spheres); and the
    packet kernel on the camera rays of one sample of each."""
    r = c3 if size == "c3_100k" else big
    n_wide = len(r.wide_nodes()[0])
    assert (n_wide <= 65536) == (size == "c3_100k"), n_wide
    case = family_stack_quantum(n_rays=10000 if size == "c3_100k" else 4000)
    bad = closest_mismatches(hc, r, case.rays)
    prims = np.ascontiguousarray(r.scene.prims)
    t0, p0 = brute_closest(hc, prims, r.generate_rays(3))
    assert (p0 >= 0).mean() > 0.5
    t, p = r.trace_kernel_packet(3); bad["packet"] = int(differ(t, p, t0, p0).sum())
    assert not _nonzero(bad), f"{size}: {bad}"


@pytest.mark.gpu
@needs_gpu
def test_gpu_scalar_tail_inside_the_closest_kernel(hc, families):
    """B2R_FLAG_REFERENCE_EXACT: the rays marked for the scalar tail (BVH.hpp:270-286) take it inside k_intersect_closest's walk, the others
    the FMA formula. The grazing family bisected against the tail test, all marked, and a random half of every other family: marked rays
    equal scalar brute force (on finite origins: the scalar tail keeps a NaN distance as its best), the others FMA brute force."""
    rs = np.random.RandomState(12)
    fails = []
    for case in [family_grazing(hc, "tail")] + families:
        n = len(case.rays)
        tail = np.ones(n, np.uint8) if case.name.startswith("grazing(tail") else rs.randint(0, 2, n).astype(np.uint8)
        r = b2r.Renderer(_scene_of(case.geometry), 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | b2r.FLAG_REFERENCE_EXACT)
        prims = np.ascontiguousarray(r.scene.prims)
        t0, p0 = brute_closest(hc, prims, case.rays); ts, ps = brute_closest(hc, prims, case.rays, scalar=True)
        t, p = r.trace_kernel_closest(case.rays, tail)
        finite = np.isfinite(case.rays[:, :3]).all(axis=1)
        on = tail.astype(bool)
        bad = {"tail": int((differ(t, p, ts, ps) & on & finite).sum()), "fma": int((differ(t, p, t0, p0) & ~on).sum())}
        assert (differ(ts, ps, t0, p0) & on & finite).sum() > 0 or not case.name.startswith("grazing(tail")   # the two formulas do differ there
        if _nonzero(bad): fails.append((case.name, bad))
        r.close()
    assert not fails, fails


# packet kernel: the camera rays cannot be injected, so the scenes are aimed at the camera rays instead
def _grazing_packet_scene(hc, r, acc, n=550, seed=13):
    """small spheres (r^2 = 1e-8 D^2, far below the leaf noise bound of 1.5e-6 D^2) 10 to 1e4 units along ~300 camera rays of sample acc
    (of 550 tried: a ray aimed at a tiny far sphere's centre can miss it in float),
    each offset perpendicular to its ray by the largest float offset hc_sphere_closest still calls a hit (bisected as in _last_hit)"""
    rs = np.random.RandomState(seed)
    rays = r.generate_rays(acc)
    geo = []
    for t in rs.choice(len(rays), n, replace=False):
        ray = np.ascontiguousarray(rays[t]); o = ray[:3].astype(np.float64); d = ray[3:].astype(np.float64)
        L = 10.0 ** rs.uniform(1, 4); rad = 1e-4 * L
        u = _unit(np.cross(d, rs.randn(3)))
        def sphere_at(off):
            s = np.zeros(1, scenes.SPHERE_DTYPE)
            s["position"] = (o + L * d + np.float64(off) * u).astype(np.float32); s["radius_sq"] = np.float32(rad * rad)
            return s
        def pred(off):
            s = sphere_at(off); s4 = np.array([*s["position"][0], s["radius_sq"][0]], np.float32)
            dd = C.c_float(); return hc.hc_sphere_closest(s4.ctypes.data, ray.ctypes.data, C.byref(dd)) == 1
        far = rad + 4.0 * np.sqrt(1.5e-6) * L
        if not pred(0.0) or pred(far): continue
        geo.append(sphere_at(_last_hit(pred, 0.0, far)))
    rest = scenes.random_scene(200, light_every=20)["geometry"]
    return np.concatenate(geo + [rest])


def _stack_under(eye, scale, n=300, seed=14):
    """spheres of radius `scale` stacked below the eye along -z, centres up to 1.6 radii off the vertical through the eye"""
    rs = np.random.RandomState(seed)
    g = np.zeros(n, scenes.SPHERE_DTYPE)
    e = np.array(eye, np.float64)
    g["position"][:, 0] = e[0] + rs.uniform(-1.6, 1.6, n) * scale; g["position"][:, 1] = e[1] + rs.uniform(-1.6, 1.6, n) * scale
    g["position"][:, 2] = e[2] - 10 * scale - 3 * scale * np.arange(n)
    g["radius_sq"] = np.float32(scale * scale)
    return g


def _packet_scene(name, hc):
    """(scene dict, frame w, h, sample indices); a scene returned as a callable is built from the camera rays of a renderer"""
    if name in ("tiny_components", "tiny_components_far_origin"):
        cam = _tiny_camera(name.endswith("far_origin"))
        sc = _scene_of(_stack_under(cam["eye"], 1e13 if name.endswith("far_origin") else 1.0)); sc["camera"] = cam
        return sc, 16, 16, range(16)
    if name == "camera_inside_a_sphere":
        sc = scenes.random_scene(2000, light_every=40)
        g = sc["geometry"]; g["position"][5] = (0, 60, 300); g["radius_sq"][5] = np.float32(900.0)   # the eye 30 units inside it ...
        g["position"][6] = (0, 60, 310); g["radius_sq"][6] = np.float32(25.0)                          # ... and inside another, off-centre
        return sc, 64, 64, [0, 7]
    if name.startswith("far_camera"):
        off = 1e4 if name.endswith("1e4") else 1e6
        sc = scenes.random_scene(3000, light_every=40); sc["geometry"] = _shifted(sc["geometry"], off)
        sc["camera"] = dict(eye=(off, off + 50, off + 2e5), dir=(0, 0, -1), focal_length=2.4e4, exposure=1.0)
        return sc, 64, 64, [0, 7]
    if name == "ties":
        geo, _, _ = family_ties()
        sc = _scene_of(geo); sc["camera"] = dict(eye=(0, 0, 70), dir=(0, 0, -1), focal_length=30.0, exposure=1.0)
        return sc, 64, 64, [0, 7]
    assert name == "grazing"
    sc = scenes.random_scene(200, light_every=20); sc["camera"] = dict(eye=(1.0, 2.0, 3.0), dir=(0.2, -0.1, -1.0), focal_length=35.0, exposure=1.0)
    return sc, 64, 64, [5]


PACKET_SCENES = ["grazing", "tiny_components", "tiny_components_far_origin", "camera_inside_a_sphere", "far_camera_1e4", "far_camera_1e6", "ties"]


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("name", PACKET_SCENES)
def test_gpu_packet_kernel_exact_on_scenes_aimed_at_camera_rays(hc, name, monkeypatch):
    """k_intersect_packet's record of every camera ray of sample acc equals brute force over b2r_generate_rays(acc). The tap runs the
    packet kernel whether or not B2R_NO_PACKET is set (the grazing scene runs with it set)."""
    if name == "grazing": monkeypatch.setenv("B2R_NO_PACKET", "1")
    else: monkeypatch.delenv("B2R_NO_PACKET", raising=False)
    sc, w, h, accs = _packet_scene(name, hc)
    r = b2r.Renderer(sc, w, h, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    if name == "grazing":   # the spheres are placed on the camera rays of this renderer's camera
        rays0 = r.generate_rays(accs[0])
        g = _scene_of(_grazing_packet_scene(hc, r, accs[0])); g["camera"] = sc["camera"]
        assert len(g["geometry"]) > 200 + 200, len(g["geometry"])
        r.SetScene(g)
        assert np.array_equal(r.generate_rays(accs[0]).view(np.uint32), rays0.view(np.uint32))
    prims = np.ascontiguousarray(r.scene.prims)
    bad, hits, n = {}, 0, 0
    for acc in accs:
        rays = r.generate_rays(acc)
        if name.startswith("tiny"):
            comp = np.abs(rays[:, 3:5]).max()
            assert comp < 2.0 ** -60 and (rays[:, 5] == -1.0).all(), comp
        t0, p0 = brute_closest(hc, prims, rays)
        t, p = r.trace_kernel_packet(acc)
        bad[acc] = int(differ(t, p, t0, p0).sum()); hits += int((p0 >= 0).sum()); n += len(rays)
    r.close()
    assert hits > 0.1 * n, (hits, n)
    assert not _nonzero(bad), f"{name}: mismatching rays per sample {_nonzero(bad)}"


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("tree", list(TREE_FLAGS) + ["sweep_fallback"])
def test_gpu_link_tables_equal_the_tree_links(tree):
    """parent[] / leaf_node[] as k_link_tables wrote them equal the links of the device tree, read on the host: after an upload, after a
    refit into the same BVH order and into a new one (leaves re-linked), and after the origin box grew (boxes refitted)."""
    if tree == "sweep_fallback":   # a hundred copies of one sphere: the sweep tree would be too deep, the packed tree is linked instead
        sc = scenes.Scene(scenes.default_scene()); d = sc["geometry"]
        sc["geometry"] = np.ascontiguousarray(np.concatenate([d, np.repeat(d[3:4], 100)]))
        flags = b2r.FLAG_GPU_TREE | b2r.FLAG_GPU_SAH
    else:
        sc = scenes.random_scene(3000, light_every=40); flags = TREE_FLAGS[tree]
    r = b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | flags)
    assert_link_tables(r, f"{tree}: upload")
    geo = np.ascontiguousarray(sc["geometry"]).copy()
    rs = np.random.RandomState(15); rad = np.sqrt(geo["radius_sq"].astype(np.float64))[:, None]
    moved = geo.copy(); moved["position"] = (geo["position"] + rs.uniform(-0.25, 0.25, (len(geo), 3)) * rad).astype(np.float32)
    r.RefitScene(moved, keep_order=True); assert_link_tables(r, f"{tree}: refit, same order")
    r.RefitScene(geo, keep_order=False); assert_link_tables(r, f"{tree}: refit, new order")
    box = r.origin_box()
    far = np.zeros((4, 6), np.float32); far[:, :3] = box[3:] + 3 * (box[3:] - box[:3]); far[:, 5] = -1
    r.trace_closest(far)
    assert not np.array_equal(r.origin_box(), box)
    assert_link_tables(r, f"{tree}: origin box grown")
    r.close()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("tree", ["default", "gpu_sweep3"])
@pytest.mark.parametrize("move", [0.25, 1.0])
def test_gpu_refit_quality_ratio_equals_the_float64_host_sum(tree, move):
    """RefitScene's quality ratio (k_tree_cost) = sum of the inner slots' half areas after the refit over the same sum as built, both read
    from wide_nodes() and summed on the host in float64 (relative 1e-6: the device adds the float terms in another order). Spheres moved by
    up to a quarter radius (DESIGN §4) and up to one radius, into the same BVH order and a new one. The eye sits inside the sphere bounds
    and the moves stay inside the origin box's slack, so the box the tree was built for is the one it is refitted for."""
    sc = scenes.random_scene(3000, light_every=40); sc["camera"] = dict(eye=(0, 50, 0), dir=(0, 0, -1), focal_length=20.0, exposure=1.0)
    rs = np.random.RandomState(16)
    for keep in (True, False):
        r = b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | TREE_FLAGS[tree])
        box = r.origin_box(); base = half_area_sum(r.wide_nodes()[0])
        geo = np.ascontiguousarray(sc["geometry"]).copy(); rad = np.sqrt(geo["radius_sq"].astype(np.float64))[:, None]
        geo["position"] = (geo["position"] + rs.uniform(-move, move, (len(geo), 3)) * rad).astype(np.float32)
        q = r.RefitScene(geo, keep_order=keep)
        assert np.array_equal(r.origin_box(), box)
        want = half_area_sum(r.wide_nodes()[0]) / base
        print(f"{tree} move {move} keep_order={keep}: quality {q:.7f}, host {want:.7f}")
        assert abs(q - want) <= 1e-6 * want, (q, want)
        assert want != 1.0
        r.close()


def _eye_rays(sc, n, seed):
    rs = np.random.RandomState(seed)
    o = np.tile(np.asarray(sc["camera"]["eye"], np.float64), (n, 1))
    d = _unit(np.c_[rs.uniform(-0.4, 0.4, n), rs.uniform(-0.4, 0.2, n), -np.ones(n)])
    return _rays(o.astype(np.float32), d.astype(np.float32))


@pytest.mark.gpu
@needs_gpu
def test_gpu_taps_leave_the_renderer_alone():
    """Accumulate 3 samples one call at a time (samples are traced ahead and wait in RAD), run every tap, accumulate 3 more and Render:
    bucket sums and frame equal those of a renderer that skipped the taps. Then the error returns of b2r_trace_kernel and
    b2r_read_link_tables."""
    sc = scenes.random_scene(5000, light_every=40)
    rays = _eye_rays(sc, 3000, 17); tfar = np.full(len(rays), 1e30, np.float32); origin = np.arange(len(rays), dtype=np.int32) % 5000
    def run(taps):
        r = b2r.Renderer(sc, 96, 64, max_bounces=6, buckets=3, flags=b2r.FLAG_FORCE_BVH, samples_in_flight=8)
        for _ in range(3): r.Accumulate(1)
        if taps:
            r.trace_kernel_closest(rays); r.trace_kernel_shadow(rays, tfar, origin); r.trace_kernel_packet(4); r.link_tables()
        for _ in range(3): r.Accumulate(1)
        assert r.Render()
        out = (r.buckets_host(), r.framebuffer.copy()); r.close()
        return out
    (ba, fa), (bb, fb) = run(True), run(False)
    assert float(ba.max()) > 0.0
    assert ba.tobytes() == bb.tobytes() and fa.tobytes() == fb.tobytes()

    L = b2r.lib(); vp = C.c_void_p
    t = np.empty(4, np.float32); p = np.empty(4, np.int32); o = np.empty(4, np.uint8); rr = np.ascontiguousarray(rays[:4]); op = np.zeros(4, np.int32)
    par = np.empty(1 << 16, np.uint32); leaf = np.empty(5000, np.uint32)
    r = b2r.Renderer(None, 64, 64, flags=b2r.FLAG_FORCE_BVH)   # no scene yet
    assert L.b2r_trace_kernel(r._h, b2r.TAP_CLOSEST, _p(rr), None, None, None, 4, 0, _p(t), _p(p), None) == b2r.ERR_STATE
    assert L.b2r_read_link_tables(r._h, _p(par), _p(leaf)) == b2r.ERR_STATE
    r.close()
    r = b2r.Renderer(sc, 64, 64, flags=b2r.FLAG_FORCE_BRUTE)
    for k in (b2r.TAP_CLOSEST, b2r.TAP_SHADOW, b2r.TAP_PACKET):
        assert L.b2r_trace_kernel(r._h, k, _p(rr), _p(tfar), _p(op), None, 4 if k != b2r.TAP_PACKET else 64 * 64, 0, _p(t), _p(p), _p(o)) == b2r.ERR_STATE
    assert L.b2r_read_link_tables(r._h, _p(par), _p(leaf)) == b2r.ERR_STATE
    r.close()
    r = b2r.Renderer(sc, 64, 64, flags=b2r.FLAG_FORCE_BVH)
    h = r._h
    assert L.b2r_trace_kernel(h, 3, _p(rr), None, None, None, 4, 0, _p(t), _p(p), None) == b2r.ERR_ARG              # unknown kernel
    assert L.b2r_trace_kernel(h, b2r.TAP_CLOSEST, None, None, None, None, 4, 0, _p(t), _p(p), None) == b2r.ERR_ARG   # no rays
    assert L.b2r_trace_kernel(h, b2r.TAP_CLOSEST, _p(rr), None, None, None, 4, 0, None, _p(p), None) == b2r.ERR_ARG   # no tfar_out
    assert L.b2r_trace_kernel(h, b2r.TAP_SHADOW, _p(rr), _p(tfar), None, None, 4, 0, None, None, _p(o)) == b2r.ERR_ARG  # no origin_prim
    assert L.b2r_trace_kernel(h, b2r.TAP_SHADOW, _p(rr), _p(tfar), _p(op), None, 4, 0, None, None, None) == b2r.ERR_ARG  # no occluded_out
    bad_op = np.array([0, 1, 5000, -1], np.int32)
    assert L.b2r_trace_kernel(h, b2r.TAP_SHADOW, _p(rr), _p(tfar), _p(bad_op), None, 4, 0, None, None, _p(o)) == b2r.ERR_ARG  # sphere 5000 of 5000
    assert L.b2r_trace_kernel(h, b2r.TAP_PACKET, None, None, None, None, 64 * 64 - 256, 0, _p(t), _p(p), None) == b2r.ERR_ARG  # n != width * height
    assert L.b2r_read_link_tables(h, None, _p(leaf)) == b2r.ERR_ARG
    r.close()


@pytest.mark.gpu
@needs_gpu
def test_gpu_tap_results_do_not_depend_on_batch_size_or_order(hc, families):
    """n = 1, 31, 33 and more than one chunk (65 536 rays): each ray's result is the one it gets in a shuffled, duplicated batch, and brute
    force's, for the closest and the shadow kernel."""
    case = families[0]
    r = b2r.Renderer(_scene_of(case.geometry), 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    prims = np.ascontiguousarray(r.scene.prims)
    rs = np.random.RandomState(18)
    pool = np.tile(case.rays, (-(-70000 // len(case.rays)), 1))[:70000]
    tf_pool = rs.uniform(1, 1000, len(pool)).astype(np.float32); op_pool = rs.randint(-1, len(prims), len(pool)).astype(np.int32)
    perm = rs.permutation(np.concatenate([np.arange(len(pool)), rs.randint(0, len(pool), 5000)]))   # shuffled, with duplicates
    ts, ps = r.trace_kernel_closest(pool[perm]); os_ = r.trace_kernel_shadow(pool[perm], tf_pool[perm], op_pool[perm])
    t0, p0 = brute_closest(hc, prims, pool); o0 = brute_any(hc, prims, pool, tf_pool)
    assert not differ(ts, ps, t0[perm], p0[perm]).any() and (os_ == o0[perm]).all()
    at = np.empty(len(pool), np.int64); at[perm[::-1]] = np.arange(len(perm))[::-1]   # where ray i of the pool first sits in the shuffled batch
    for n in (1, 31, 33, 70000):
        t, p = r.trace_kernel_closest(pool[:n]); o = r.trace_kernel_shadow(pool[:n], tf_pool[:n], op_pool[:n])
        assert not differ(t, p, ts[at[:n]], ps[at[:n]]).any(), n
        assert (o == os_[at[:n]]).all(), n
    r.close()
