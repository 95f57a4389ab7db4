"""The closest-hit walk of secondary rays starts at the node that holds the sphere the ray leaves from and climbs (TravClosestT, b2r_shade.h):
k_shade queues the start node with every path it continues (QueueDev::N), k_intersect_closest reads it. The walk is exact from any start
node of the tree it walks: these tests hold it to brute force on the adversarial ray families of tests/test_traversal_exact.py.

CPU tier: tests/climbcheck/climb_taps.cpp (the host check, unchanged, plus cc_trace_closest: the kernels' TravClosestT started at a leaf's
node and climbing through parent[]), compiled with g++ into a temporary directory, on every family and every tree kind. GPU tier (-m gpu):
k_intersect_closest through b2r_trace_kernel with start nodes at every leaf, for every tree flag and after refits, with the shared-memory
stack spilling, in the counting and the B2R_FLAG_REFERENCE_EXACT instantiations; and frames enqueued back to back across scene changes and
refits, against a renderer that waits after every call and against brute force."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import b2r
import scenes
from conftest import have_gpu
import test_traversal_exact as tx
from test_traversal_kernels import _nest_case, _nest_scene, _renderer, brute_closest, differ, shadow_batch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
needs_gpu = pytest.mark.skipif(not have_gpu(), reason="needs a CUDA device")
_CLIMBTAPS = None


def climbtaps():
    """tests/climbcheck/climb_taps.cpp (+ csrc/b2r_host.cpp) compiled once per session into a temporary directory with the host check's flags"""
    global _CLIMBTAPS
    if _CLIMBTAPS is None:
        import tempfile
        csrc = os.path.join(ROOT, "cpu-raytracing-experiments_b200", "csrc")
        out = os.path.join(tempfile.mkdtemp(prefix="b2r_climbtaps_"), "libclimbtaps.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mavx2", "-mfma", "-fPIC", "-shared", "-I/usr/local/cuda/include", "-I", csrc,
                               os.path.join(HERE, "climbcheck", "climb_taps.cpp"), os.path.join(csrc, "b2r_host.cpp"), "-o", out])
        L = tx._declare(C.CDLL(out))
        vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int
        L.cc_trace_closest.argtypes = [i32, vp, vp, u32, vp, u32, vp, vp, u32, i32, vp, vp, vp, vp]; L.cc_trace_closest.restype = i32
        _CLIMBTAPS = L
    return _CLIMBTAPS


@pytest.fixture(scope="module")
def cc():
    return climbtaps()


@pytest.fixture(scope="module")
def hc(hostcheck):
    return tx._declare(hostcheck)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def host_closest_climb(cc, case, kind, origin, tail=False, counts=None):
    n = len(case.rays); t = np.empty(n, np.float32); p = np.empty(n, np.int32)
    prims, moved = (tx._moved_copy(case.prims), case.prims) if kind == tx.KINDS["refit"] else (case.prims, None)
    rc = cc.cc_trace_closest(kind, _p(prims), _p(case.nodes), len(case.nodes), _p(moved), len(case.prims), _p(case.box6), _p(case.rays), n, int(tail),
                             _p(origin), _p(t), _p(p), _p(counts))
    return rc, t, p


def every_leaf(case):
    """the family's rays, and as many copies as it takes for the walks between them to start at every sphere once (BVH order), and from the root"""
    n, m = len(case.rays), len(case.prims)
    k = -(-m // n)
    cover = np.random.RandomState(m).permutation(np.arange(k * n) % m)
    origin = np.concatenate([case.origin_prim, np.full(n, -1), cover]).astype(np.int32)
    c = tx.Case(case.name, case.geometry, np.tile(case.rays, (k + 2, 1)), box6=case.box6, tail=case.tail)
    return c, origin


def climb_mismatches(cc, case):
    """{(walk, tree kind): rays whose climbing walk differs from brute force} over every tree kind, with and without the scalar tail"""
    case, origin = every_leaf(case)
    t0, p0, ts0, ps0, _ = tx.brute(cc, case)
    finite = np.isfinite(case.rays[:, :3]).all(axis=1)
    bad = {}
    for name, kind in tx.KINDS.items():
        rc, t, p = host_closest_climb(cc, case, kind, origin)
        if rc == 1: continue  # a sweep tree too deep for kTraversalStack: the library builds the packed tree instead
        assert rc == 0, (case.name, name, rc)
        bad[("closest_climb", name)] = int(differ(t, p, t0, p0).sum())
        if case.tail:
            rc, t, p = host_closest_climb(cc, case, kind, origin, tail=True); assert rc == 0
            bad[("closest_climb_tail", name)] = int((differ(t, p, ts0, ps0) & finite).sum())
    return {k: v for k, v in bad.items() if v}


# ------------------------------------------------------------------------------------------------ CPU tier
def _cpu_families(hc):
    yield from (tx.family_directions(o, l) for o, l in [(0.0, 400.0), (0.0, 3e4), (1e4, 400.0), (1e6, 2e5)])
    yield from (tx.family_grazing(hc, t, o) for t in ("closest", "tail") for o in (0.0, 1e4))
    yield from (c for c in (tx.family_box_features(hc, k) for k in tx.KINDS.values()) if c is not None)
    yield tx.ties_case(hc)
    yield tx.family_origins()


def test_climbing_closest_walk_equals_brute_force_on_every_family(hc, cc):
    """Every family of test_traversal_exact through every tree kind, each ray's walk started at its own origin sphere, at the root and, in
    copies, at every sphere of the tree: prim ids and tfar bits equal brute force (the scalar tail: scalar brute force, finite origins)."""
    fails = []
    for case in _cpu_families(hc):
        bad = climb_mismatches(cc, case)
        if bad: fails.append((case.name, bad))
    assert not fails, fails


def test_climbing_closest_walk_at_100k_spheres(cc):
    """C3's 100k spheres, where the stack entries keep 8 mantissa bits: walks from the rays' random origin spheres equal brute force for
    every tree kind, and a walk from the root (start -1) is the plain root walk of hc_trace_closest, node for node."""
    case = tx.family_stack_quantum(n_rays=4000)
    t0, p0, _, _, _ = tx.brute(cc, case)
    bad = {}
    for name, kind in tx.KINDS.items():
        rc, t, p = host_closest_climb(cc, case, kind, case.origin_prim)
        if rc == 1: continue
        assert rc == 0, (name, rc)
        bad[name] = int(differ(t, p, t0, p0).sum())
    assert not any(bad.values()), bad
    n = len(case.rays); root = np.full(n, -1, np.int32)
    c_root = np.zeros(3 * n, np.uint32); c_none = np.zeros(3 * n, np.uint32)
    assert host_closest_climb(cc, case, tx.KINDS["sah"], root, counts=c_root)[0] == 0
    assert host_closest_climb(cc, case, tx.KINDS["sah"], None, counts=c_none)[0] == 0
    assert np.array_equal(c_root, c_none)
    rc, t, p = tx.host_closest(cc, case, tx.KINDS["sah"])
    assert rc == 0 and not differ(t, p, t0, p0).any()


def test_climb_tap_rejects_an_origin_sphere_out_of_range(cc):
    case = tx.family_origins()
    origin = np.zeros(len(case.rays), np.int32); origin[7] = len(case.prims)
    assert host_closest_climb(cc, case, tx.KINDS["sah"], origin)[0] == b2r.ERR_ARG


# ------------------------------------------------------------------------------------------------ GPU tier
def kernel_mismatches(hc, r, case, tail=None):
    """rays where k_intersect_closest, started at each ray's own origin sphere, at the root and (in copies) at every sphere of the renderer's
    BVH order, differs from brute force over the renderer's spheres. tail: mark a random half of the rays for the scalar tail (EXACT)."""
    rays, _, origin = shadow_batch(case, r)
    prims = np.ascontiguousarray(r.scene.prims)
    t0, p0 = brute_closest(hc, prims, rays)
    if tail is None:
        t, p = r.trace_kernel_closest(rays, origin_prim=origin)
        return int(differ(t, p, t0, p0).sum())
    mark = np.random.RandomState(len(rays)).randint(0, 2, len(rays)).astype(np.uint8); on = mark.astype(bool)
    ts, ps = brute_closest(hc, prims, rays, scalar=True)
    finite = np.isfinite(rays[:, :3]).all(axis=1)
    t, p = r.trace_kernel_closest(rays, tail=mark, origin_prim=origin)
    return int((differ(t, p, ts, ps) & on & finite).sum() + (differ(t, p, t0, p0) & ~on).sum())


@pytest.fixture(scope="module")
def families(hc):
    return tx._gpu_cases(hc)


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("tree", list(tx.TREE_FLAGS) + ["refit", "refit_keep"])
def test_gpu_closest_kernel_climbs_exactly_from_every_leaf(hc, families, tree):
    """k_intersect_closest with start nodes at every leaf, for every tree flag and after a refit into a new BVH order (k_link_tables runs
    again) and into the same one; family 3 aims at the device tree's own slot boxes."""
    fails = []
    sc = tx._scene_of(scenes.random_scene(1500, light_every=50)["geometry"])
    r = _renderer(sc, tree)
    case = tx._gpu_feature_case(r, sc["geometry"])
    bad = kernel_mismatches(hc, r, case)
    if bad: fails.append((case.name, bad))
    r.close()
    for case in families:
        r = _renderer(tx._scene_of(case.geometry), tree)
        bad = kernel_mismatches(hc, r, case)
        if bad: fails.append((case.name, bad))
        r.close()
    assert not fails, f"tree {tree}: {fails}"


@pytest.mark.gpu
@needs_gpu
def test_gpu_climbing_closest_kernel_deep_stack_count_and_exact_instantiations(hc, families):
    """The climbing walk with the shared-memory stack spilling (nested spheres), in the B2R_FLAG_COUNT_TESTS instantiation, and in the
    B2R_FLAG_REFERENCE_EXACT instantiation with the scalar tail on a random half of the rays; an origin sphere out of range is refused."""
    sc = _nest_scene()
    r = b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH)
    assert r.wide_nodes()[1] > 13
    case = _nest_case(sc)
    bad = {}
    for flags in (b2r.FLAG_FORCE_BVH, b2r.FLAG_FORCE_BVH | b2r.FLAG_COUNT_TESTS):
        r.set_flags(flags); bad[(flags, "nest")] = kernel_mismatches(hc, r, case)
    out = np.full(len(case.rays), -1, np.int32); out[3] = len(r.scene.prims)
    with pytest.raises(b2r.B2RError):
        r.trace_kernel_closest(case.rays, origin_prim=out)
    r.close()
    r = b2r.Renderer(sc, 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | b2r.FLAG_REFERENCE_EXACT)   # (chosen at creation only)
    bad[("exact", "nest")] = kernel_mismatches(hc, r, case, tail=True)
    r.close()
    for case in families:
        r = b2r.Renderer(tx._scene_of(case.geometry), 64, 64, max_bounces=4, buckets=1, flags=b2r.FLAG_FORCE_BVH | b2r.FLAG_REFERENCE_EXACT)
        bad[("exact", case.name)] = kernel_mismatches(hc, r, case, tail=True)
        r.close()
    bad = {k: v for k, v in bad.items() if v}
    assert not bad, bad


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("tree", ["default", "gpu_sweep3"])
def test_gpu_frames_back_to_back_across_scene_changes_and_refits(tree):
    """Start nodes never outlive the tree they were read from: frames enqueued back to back (no host wait) across uploads of other scenes —
    a smaller one, whose tree has fewer nodes than the start nodes of the frame before could name — and refits into a new BVH order. Every
    frame must equal the same frame of a renderer that waits after every call, and brute force."""
    w, h, mb, K = 160, 96, 8, 2
    big = scenes.random_scene(6000, light_every=40)
    small = scenes.random_scene(700, light_every=20, seed=0x1234567)
    rs = np.random.RandomState(3)
    def moved(geo):
        out = geo.copy(); r = np.sqrt(out["radius_sq"])
        out["position"] += (rs.uniform(-1, 1, (len(out), 3)) * (0.6 * r)[:, None]).astype(np.float32)
        idx = rs.choice(len(out), len(out) // 20, replace=False)   # some spheres jump anywhere: the refit re-links leaves into a new order
        out["position"][idx] = rs.uniform(geo["position"].min(0), geo["position"].max(0), (len(idx), 3)).astype(np.float32)
        return out
    geo1 = moved(big["geometry"]); geo2 = moved(geo1); geo3 = moved(small["geometry"])
    plan = ["big", "refit1", "small", "big", "refit2", "small", "refit3", "big"]
    flags = b2r.FLAG_FORCE_BVH | tx.TREE_FLAGS[tree]
    def drive(r, steps, wait):
        out = []
        for step in steps:
            if step == "refit1": r.RefitScene(geo1, want_quality=False)
            elif step == "refit2": r.RefitScene(geo2, want_quality=False)
            elif step == "refit3": r.RefitScene(geo3, want_quality=False)
            else: r.SetScene(b2r.PreparedScene(big if step == "big" else small, w, h))
            r.ResetAccumulator(); r.Accumulate(2 * K)
            if wait: assert r.Render(); out.append(r.buckets_host().copy())
            else: assert r.RenderDevice()
        return out
    a = b2r.Renderer(big, w, h, max_bounces=mb, buckets=K, flags=flags); want = drive(a, plan, True); a.close()
    b = b2r.Renderer(big, w, h, max_bounces=mb, buckets=K, flags=b2r.FLAG_FORCE_BRUTE); ref = drive(b, plan, True); b.close()
    for i in range(len(plan)):
        assert want[i].tobytes() == ref[i].tobytes(), f"step {i} ({plan[i]}): BVH differs from brute force"
        assert float(want[i].max()) > 0.0
    for upto in (3, 5, 6, len(plan)):   # drained after prefixes that end on a smaller scene, a refit and a larger scene
        r = b2r.Renderer(big, w, h, max_bounces=mb, buckets=K, flags=flags)
        drive(r, plan[:upto], False); r.sync()
        assert r.buckets_host().tobytes() == want[upto - 1].tobytes(), f"pipelined run ending on step {upto - 1} ({plan[upto - 1]}) differs"
        r.close()
