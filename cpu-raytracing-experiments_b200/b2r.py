"""ctypes binding of libb2r.so (include/b2r.h) plus a Python mirror of the reference's Renderer interface.

The reference is a C++ class template used directly by its app (Renderer.hpp:28-479, call sites Application.cpp:373-382);
the C++ mirror lives in host/Renderer.hpp. This module is the same surface for the Python test and bench harness:

    scene = PreparedScene(scenes.default_scene(), width, height)   # BVH (BVH.hpp:90-206) + lights (Scene.hpp:12-16) + camera
    r = Renderer(scene, width, height)                              # Renderer(const Scene&) + Resize
    r.Accumulate(); ...; r.Render()                                 # Renderer.hpp:73, :436
    r.framebuffer                                                   # (H, W, 4) float32, row 0 = y 0

There is no CPU fallback: importing works anywhere (so symbols can be checked on a CPU box), creating a Renderer without a
CUDA device raises B2RError.
"""
import ctypes as C
import os

import numpy as np

try:
    from . import scenes as _scenes
except ImportError:  # imported as a top-level module from the package directory
    import scenes as _scenes

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2R_LIB_PATH", os.path.join(_HERE, "libb2r.so"))  # override: kernel A/B experiments only

FLAG_FORCE_BRUTE, FLAG_FORCE_BVH, FLAG_NO_MIS, FLAG_COUNT_TESTS, FLAG_NO_GRAPH, FLAG_REFERENCE_TREE, FLAG_REFERENCE_EXACT, FLAG_NO_SPECULATION, FLAG_GPU_TREE = 1, 2, 4, 8, 16, 32, 64, 128, 256
FLAG_GPU_SAH = 1024  # with FLAG_GPU_TREE: the sweep tree (SAH cuts along the curve order) instead of the packed one
FLAG_GPU_SAH3 = 2048  # with FLAG_GPU_TREE: the three-axis sweep tree (full-sweep SAH over the x, y, z orders)
FLAG_GGX = 512  # the reference's `#define BRDF 1` closure (Closure<GGX>, DataStreams.hpp:184-219)
FLAG_DIELECTRIC = 4096  # materials with max(transmission) > 0 render as smooth dielectrics of IOR 1 + IOR_minus_one (DESIGN.md §2)
FLAG_SKY_LIGHT = 8192  # the HDRI sky sampled as a light, MIS-combined with the BSDF-sampled misses (DESIGN.md §2)
FLAG_LIGHT_TREE = 16384  # sphere lights picked by importance from a light tree instead of uniformly (DESIGN.md §2)
TAP_CLOSEST, TAP_SHADOW, TAP_PACKET = 0, 1, 2  # b2r_trace_kernel: which traversal kernel of a frame runs
OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_NO_LIGHTS, ERR_BVH, NOT_READY = 0, -1, -2, -3, -4, -5, 1
KERNEL_KINDS = ["generate", "bounce_brute", "intersect_closest", "shade", "intersect_shadow", "accumulate", "resolve"]
COUNTER_NAMES = ["extension_rays", "shadow_rays", "shaded_hits", "terminated", "dropped", "sphere_tests", "box_tests", "launches", "radiance_events", "reserved"]

# every symbol include/b2r.h declares (tests/test_abi.py checks the header against this list and the library against both)
ABI_SYMBOLS = [
    "b2r_bvh_build", "b2r_bvh_build_ex", "b2r_find_lights", "b2r_camera_lookat", "b2r_camera_ray", "b2r_create", "b2r_destroy", "b2r_resize", "b2r_reset", "b2r_set_stream",
    "b2r_sync", "b2r_upload_scene", "b2r_refit_scene", "b2r_set_camera", "b2r_set_lens", "b2r_accumulate", "b2r_resolve", "b2r_resolve_async", "b2r_resolve_device", "b2r_frame_wait", "b2r_resolve_from", "b2r_ipc_export_buckets", "b2r_ipc_open_peers", "b2r_ipc_close", "b2r_resolve_peers", "b2r_team_export", "b2r_team_open", "b2r_team_resolve", "b2r_team_error", "b2r_team_close", "b2r_host_register", "b2r_host_unregister", "b2r_get_accumulations", "b2r_set_accumulations",
    "b2r_read_buckets", "b2r_write_buckets", "b2r_save_checkpoint", "b2r_load_checkpoint", "b2r_device_buckets", "b2r_device_framebuffer", "b2r_read_counters", "b2r_reset_counters", "b2r_read_bounce_counts",
    "b2r_read_kernel_times", "b2r_set_flags", "b2r_generate_rays", "b2r_trace_closest", "b2r_trace_shadow", "b2r_trace_kernel", "b2r_read_wide_nodes", "b2r_read_link_tables", "b2r_read_sky_tables", "b2r_read_light_tree", "b2r_get_origin_box",
    "b2r_write_hdr", "b2r_read_hdr", "b2r_last_error", "b2r_abi_version",
]


class B2RError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"libb2r error {code}: {text}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("max_bounces", C.c_uint32), ("buckets", C.c_uint32), ("flags", C.c_uint32),
                ("device", C.c_int32), ("bucket_first", C.c_uint32), ("bucket_stride", C.c_uint32), ("samples_in_flight", C.c_uint32)]


_lib = None


def lib():
    """Load libb2r.so (built in-tree by __graft_entry__.build()). Fails loudly when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2RError(ERR_STATE, f"{LIB_PATH} not built - run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(LIB_PATH)
        vp, u32, i32, f32 = C.c_void_p, C.c_uint32, C.c_int32, C.c_float
        sig = {
            "b2r_bvh_build": [vp, u32, vp, vp, vp, vp], "b2r_bvh_build_ex": [vp, u32, u32, f32, vp, vp, vp, vp], "b2r_find_lights": [vp, u32, vp, u32, vp, vp],
            "b2r_camera_lookat": [vp, vp, u32, u32, f32, f32, vp], "b2r_camera_ray": [vp, vp, f32, f32, f32, i32, i32, vp, vp, vp], "b2r_create": [vp, vp], "b2r_resize": [vp, u32, u32], "b2r_reset": [vp],
            "b2r_set_stream": [vp, vp], "b2r_sync": [vp],
            "b2r_upload_scene": [vp, vp, vp, u32, u32, vp, u32, vp, u32, vp, u32, vp, vp, i32, i32],
            "b2r_refit_scene": [vp, vp, u32, vp, u32, vp, u32, vp, u32, vp],
            "b2r_set_camera": [vp, vp, vp, f32, f32, f32, f32], "b2r_set_lens": [vp, f32, f32], "b2r_accumulate": [vp, u32], "b2r_resolve": [vp, vp, C.c_int], "b2r_resolve_async": [vp, vp, C.c_int], "b2r_resolve_device": [vp, C.c_int], "b2r_frame_wait": [vp], "b2r_resolve_from": [vp, vp, vp, C.c_int], "b2r_ipc_export_buckets": [vp, vp], "b2r_ipc_open_peers": [vp, vp, u32, u32], "b2r_ipc_close": [vp], "b2r_resolve_peers": [vp, vp, C.c_int], "b2r_team_export": [vp, vp], "b2r_team_open": [vp, vp, u32, u32], "b2r_team_resolve": [vp, vp, C.c_int, C.c_int], "b2r_team_error": [vp, vp], "b2r_team_close": [vp],
            "b2r_host_register": [vp, C.c_size_t], "b2r_host_unregister": [vp], "b2r_get_accumulations": [vp, vp], "b2r_set_accumulations": [vp, u32], "b2r_read_buckets": [vp, vp], "b2r_write_buckets": [vp, vp],
            "b2r_device_buckets": [vp, vp, vp], "b2r_device_framebuffer": [vp, vp, vp], "b2r_read_counters": [vp, vp], "b2r_reset_counters": [vp], "b2r_read_bounce_counts": [vp, vp, vp, u32],
            "b2r_read_kernel_times": [vp, vp, vp, C.c_int], "b2r_set_flags": [vp, u32], "b2r_generate_rays": [vp, u32, vp],
            "b2r_save_checkpoint": [vp, C.c_char_p], "b2r_load_checkpoint": [vp, C.c_char_p], "b2r_write_hdr": [C.c_char_p, vp, u32, u32], "b2r_read_hdr": [C.c_char_p, vp, vp, vp], "b2r_trace_closest": [vp, vp, u32, vp, vp], "b2r_trace_shadow": [vp, vp, vp, u32, vp], "b2r_trace_kernel": [vp, C.c_int, vp, vp, vp, vp, u32, u32, vp, vp, vp], "b2r_read_wide_nodes": [vp, vp, vp, vp], "b2r_read_link_tables": [vp, vp, vp], "b2r_read_sky_tables": [vp, vp, vp, vp, vp, vp], "b2r_read_light_tree": [vp, vp, vp, vp], "b2r_get_origin_box": [vp, vp],
        }
        for name, args in sig.items():
            fn = getattr(L, name); fn.argtypes = args; fn.restype = C.c_int
        L.b2r_destroy.argtypes = [vp]; L.b2r_destroy.restype = None
        L.b2r_last_error.restype = C.c_char_p; L.b2r_abi_version.restype = C.c_int
        _lib = L
    return _lib


def _check(rc):
    if rc < 0:
        raise B2RError(rc, lib().b2r_last_error().decode())
    return rc


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


def build_bvh(geometry, log_cluster_size=0, cost_ratio=1.0):
    """BoundingVolumeHierarchy<Sphere>(geometry, SplitHeuristic{log_cluster_size, cost_ratio}) — BVH.hpp:70-83,90-206. Returns (nodes, prims, prim_ids)."""
    geo = np.ascontiguousarray(geometry, dtype=_scenes.SPHERE_DTYPE); n = len(geo)
    nodes = np.zeros(max(1, 2 * n - 1), _scenes.NODE_DTYPE); prims = np.zeros(n, _scenes.SPHERE_DTYPE); ids = np.zeros(n, np.uint32)
    nn = C.c_uint32(0)
    _check(lib().b2r_bvh_build_ex(_ptr(geo), n, log_cluster_size, cost_ratio, _ptr(nodes), _ptr(prims), _ptr(ids), C.addressof(nn)))
    return nodes[:nn.value], prims, ids


def find_lights(geometry, material):
    """LightingAcceleration(geometry, material) — Scene.hpp:12-16."""
    geo = np.ascontiguousarray(geometry, dtype=_scenes.SPHERE_DTYPE); mat = np.ascontiguousarray(material, dtype=_scenes.MATERIAL_DTYPE)
    out = np.zeros(len(geo), np.int32); n = C.c_uint32(0)
    _check(lib().b2r_find_lights(_ptr(geo), len(geo), _ptr(mat), len(mat), _ptr(out), C.addressof(n)))
    return out[:n.value].copy()


def camera_lookat(eye, direction, width, height, focal_length, exposure=1.0):
    """Camera{eye, dir, w, h, focal} + Resize — Camera.hpp:21-32,47-50,61-68. Returns the 11 floats of b2r_set_camera."""
    out = np.zeros(11, np.float32)
    e = np.asarray(eye, np.float32); d = np.asarray(direction, np.float32)
    _check(lib().b2r_camera_lookat(_ptr(e), _ptr(d), width, height, focal_length, exposure, _ptr(out)))
    return out


class PreparedScene:
    """Scene (Scene.hpp:19-26) with acceleration_structure and lighting_acceleration built, as Application.cpp:233-234 does."""

    def __init__(self, scene, width, height):
        self.scene = scene
        self.geometry = np.ascontiguousarray(scene["geometry"], dtype=_scenes.SPHERE_DTYPE)
        self.material = np.ascontiguousarray(scene["material"], dtype=_scenes.MATERIAL_DTYPE)
        self.nodes, self.prims, self.prim_ids = build_bvh(self.geometry)
        self.lights = find_lights(self.geometry, self.material)
        self.ambient = np.asarray(scene["ambient"], np.float32)
        self.hdri = None if scene.get("hdri") is None else np.ascontiguousarray(scene["hdri"], np.float32)
        self.set_view(width, height)

    def set_view(self, width, height):
        cam = self.scene["camera"]
        self.camera = camera_lookat(cam["eye"], cam["dir"], width, height, cam["focal_length"], cam["exposure"])


class Renderer:
    """Renderer<Policy> (Renderer.hpp:28-479) on one B200. Method names follow the reference."""

    TileRoot = 16

    @staticmethod
    def RequiredTiling():
        return 16  # Renderer.hpp:36

    def __init__(self, scene, width, height, max_bounces=16, buckets=5, flags=0, device=0, bucket_first=0, bucket_stride=0,
                 samples_in_flight=0, stream=None):
        self._h = C.c_void_p(None)
        cfg = Config(width, height, max_bounces, buckets, flags, device, bucket_first, bucket_stride, samples_in_flight)
        _check(lib().b2r_create(C.byref(self._h), C.byref(cfg)))
        self.width, self.height, self.max_bounces, self.buckets, self.flags = width, height, max_bounces, buckets, flags
        self.h_tiles, self.v_tiles = width // 16, height // 16
        self.framebuffer = np.zeros((height, width, 4), np.float32)
        if stream is not None:
            _check(lib().b2r_set_stream(self._h, C.c_void_p(stream)))
        self.scene = None
        if scene is not None:
            self.SetScene(scene)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().b2r_destroy(self._h); self._h = C.c_void_p(None)

    __del__ = close

    # -- scene / camera (the reference holds `const Scene&`; edits are re-uploaded explicitly, cf. Application.cpp:508-510)
    def SetScene(self, ps):
        if not isinstance(ps, PreparedScene):
            ps = PreparedScene(ps, self.width, self.height)
        self.scene = ps
        hd = ps.hdri
        _check(lib().b2r_upload_scene(self._h, _ptr(ps.prims), _ptr(ps.nodes), len(ps.prims), len(ps.nodes), _ptr(ps.material), len(ps.material),
                                      _ptr(ps.lights), len(ps.lights), _ptr(ps.geometry), len(ps.geometry), _ptr(ps.ambient),
                                      _ptr(hd), 0 if hd is None else hd.shape[1], 0 if hd is None else hd.shape[0]))
        self.SetCamera(ps.camera)

    def RefitScene(self, geometry, material=None, want_quality=True, keep_order=False):
        """Scene edit without rebuilding the traversal tree (cf. Application.cpp:508-510): `geometry` holds the moved spheres in ORIGINAL
        order, same count as the scene set before. As the reference does after an edit, the reference BVH is rebuilt on the host
        (BoundingVolumeHierarchy ctor: new leaf order, Q6/Q9 depend on it) and the light list re-derived; the GPU keeps the traversal
        tree's topology, re-links its leaves to the new order and recomputes its boxes (b2r_refit_scene). keep_order=True skips the
        host rebuild and keeps the previous leaf order. Returns the tree-quality ratio (1.0 = as built) or None. The caller resets the
        accumulator."""
        import copy
        geo = np.ascontiguousarray(geometry, dtype=_scenes.SPHERE_DTYPE)
        if self.scene is None or len(geo) != len(self.scene.geometry):
            raise B2RError(ERR_ARG, "RefitScene keeps the sphere count of the scene set before")
        ps = self.scene = copy.copy(self.scene)  # the caller's PreparedScene stays as it was
        if material is not None:
            ps.material = np.ascontiguousarray(material, dtype=_scenes.MATERIAL_DTYPE)
        ps.geometry = geo
        if keep_order:
            ps.prims = np.ascontiguousarray(geo[ps.prim_ids])
        else:
            ps.nodes, ps.prims, ps.prim_ids = build_bvh(geo)
        ps.lights = find_lights(ps.geometry, ps.material)
        q = C.c_float(0.0)
        _check(lib().b2r_refit_scene(self._h, _ptr(ps.prims), len(ps.prims), _ptr(ps.material), len(ps.material), _ptr(ps.lights), len(ps.lights),
                                     _ptr(ps.geometry), len(ps.geometry), C.addressof(q) if want_quality else None))
        return q.value if want_quality else None

    def SetCamera(self, cam11):
        cam = np.ascontiguousarray(cam11, np.float32)
        self._cam = cam
        _check(lib().b2r_set_camera(self._h, _ptr(cam[0:3]), _ptr(cam[3:7]), float(cam[7]), float(cam[8]), float(cam[9]), float(cam[10])))

    def SetLens(self, radius, focus_distance):
        """Thin-lens depth of field (b2r_set_lens): lens radius and focus distance in scene units (the caller converts the app's
        Projection::aperture_radius, which is in mm); the plane at focus_distance along the view direction is sharp. radius 0 = the
        pinhole camera, bit for bit. Takes effect from the next Accumulate, like SetCamera."""
        _check(lib().b2r_set_lens(self._h, float(radius), float(focus_distance)))

    # -- Renderer.hpp:53-67
    def Resize(self, width, height):
        _check(lib().b2r_resize(self._h, width, height))
        self.width, self.height, self.h_tiles, self.v_tiles = width, height, width // 16, height // 16
        self.framebuffer = np.zeros((height, width, 4), np.float32)
        if self.scene is not None:
            self.scene.set_view(width, height); self.SetCamera(self.scene.camera)

    def ResetAccumulator(self):
        _check(lib().b2r_reset(self._h))

    @property
    def accumulations(self):
        v = C.c_uint32(0); _check(lib().b2r_get_accumulations(self._h, C.byref(v))); return v.value

    @accumulations.setter
    def accumulations(self, v):
        _check(lib().b2r_set_accumulations(self._h, v))

    # -- the hot path
    def Accumulate(self, n=1):
        """Renderer::Accumulate() n times (Renderer.hpp:73-434). Asynchronous."""
        _check(lib().b2r_accumulate(self._h, n))

    def Render(self, tonemap=True, out=None, to_host=True, dev_buckets=None):
        """Renderer::Render() (Renderer.hpp:436-478). Returns False (and leaves framebuffer untouched) unless accumulations % K == 0.
        to_host=False leaves the RGBA32F frame on the device; dev_buckets reads the bucket sums from another device array
        (the NCCL-combined buckets of a multi-GPU frame)."""
        dst = (self.framebuffer if out is None else out) if to_host else None
        rc = _check(lib().b2r_resolve_from(self._h, C.c_void_p(dev_buckets) if dev_buckets else None, _ptr(dst), 1 if tonemap else 0))
        return rc == OK

    def RenderAsync(self, out, tonemap=True):
        """Render() without the stall (b2r_resolve_async): the frame is copied to `out` (page-locked numpy array) on a second stream while
        the next Accumulate calls run; WaitFrame() blocks until it has landed. Returns False when accumulations % K != 0."""
        return _check(lib().b2r_resolve_async(self._h, _ptr(out), 1 if tonemap else 0)) == OK

    def RenderDevice(self, tonemap=True):
        """Render() into the device framebuffer without waiting (b2r_resolve_device): frames enqueued back to back are pipelined on the device.
        sync() before the frame is read. Returns False when accumulations % K != 0."""
        return _check(lib().b2r_resolve_device(self._h, 1 if tonemap else 0)) == OK

    def WaitFrame(self):
        _check(lib().b2r_frame_wait(self._h))

    # -- multi-GPU fused resolve over peer memory (see b2r_dist.open_peers)
    def ipc_export_buckets(self):
        h = (C.c_ubyte * 64)(); _check(lib().b2r_ipc_export_buckets(self._h, h)); return bytes(h)

    def ipc_open_peers(self, handles, my_rank):
        blob = b"".join(handles); buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        _check(lib().b2r_ipc_open_peers(self._h, buf, len(handles), my_rank))

    def ipc_close(self):
        _check(lib().b2r_ipc_close(self._h))

    def RenderPeers(self, tonemap=True, out=None, to_host=True):
        """Render() reading every bucket from its owner GPU over NVLink (after ipc_open_peers and a barrier)."""
        dst = (self.framebuffer if out is None else out) if to_host else None
        return _check(lib().b2r_resolve_peers(self._h, _ptr(dst), 1 if tonemap else 0)) == OK

    # -- team mode: multi-GPU frame without host barriers (see b2r_dist.open_team)
    def team_export(self):
        h = (C.c_ubyte * 192)(); _check(lib().b2r_team_export(self._h, h)); return bytes(h)

    def team_open(self, handles, my_rank):
        blob = b"".join(handles); buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        _check(lib().b2r_team_open(self._h, buf, len(handles), my_rank))

    def team_close(self):
        _check(lib().b2r_team_close(self._h))

    def RenderTeam(self, tonemap=True, out=None, to_host=True, use_async=False):
        """Render() of a multi-GPU frame, called by every rank: this rank resolves its slab of tiles (buckets read from their owners over
        NVLink) into rank 0's framebuffer; rank 0 copies the frame to `out` / self.framebuffer (use_async: on its copy stream, WaitFrame()
        to join). No host synchronisation between ranks."""
        dst = (self.framebuffer if out is None else out) if to_host else None
        return _check(lib().b2r_team_resolve(self._h, _ptr(dst), 1 if tonemap else 0, 1 if use_async else 0)) == OK

    def team_error(self):
        v = C.c_uint32(0); _check(lib().b2r_team_error(self._h, C.byref(v))); return v.value

    def GetFrame(self):
        return self.framebuffer  # Renderer.hpp:68 returns the Vulkan Image; here: the host RGBA32F array

    # -- taps
    def sync(self):
        _check(lib().b2r_sync(self._h))

    def buckets_host(self):
        out = np.empty((self.buckets, 3, self.width * self.height), np.float32); _check(lib().b2r_read_buckets(self._h, _ptr(out))); return out

    def write_buckets(self, arr):
        a = np.ascontiguousarray(arr, np.float32); _check(lib().b2r_write_buckets(self._h, _ptr(a)))

    def SaveCheckpoint(self, path):
        """Bucket sums + sample counter as one file (b2r_save_checkpoint); LoadCheckpoint on a renderer of the same configuration resumes the
        same image bit for bit."""
        _check(lib().b2r_save_checkpoint(self._h, str(path).encode()))

    def LoadCheckpoint(self, path):
        _check(lib().b2r_load_checkpoint(self._h, str(path).encode()))

    def device_buckets(self):
        p = C.c_void_p(None); n = C.c_size_t(0); _check(lib().b2r_device_buckets(self._h, C.byref(p), C.byref(n))); return p.value, n.value

    def device_framebuffer(self):
        p = C.c_void_p(None); n = C.c_size_t(0); _check(lib().b2r_device_framebuffer(self._h, C.byref(p), C.byref(n))); return p.value, n.value

    def counters(self):
        out = (C.c_uint64 * 10)(); _check(lib().b2r_read_counters(self._h, out)); return dict(zip(COUNTER_NAMES, out[:]))

    def bounce_counts(self):
        """(paths, shadow): extension rays entering each bounce and shadow rays queued at each bounce of the last wavefront batch."""
        n = self.max_bounces + 1; a = np.zeros(n, np.uint32); b = np.zeros(n, np.uint32)
        _check(lib().b2r_read_bounce_counts(self._h, _ptr(a), _ptr(b), n)); return a, b

    def reset_counters(self):
        _check(lib().b2r_reset_counters(self._h))

    def kernel_times(self, reset=True):
        ms = (C.c_double * 8)(); n = (C.c_uint64 * 8)(); _check(lib().b2r_read_kernel_times(self._h, ms, n, 1 if reset else 0))
        return {k: (ms[i], n[i]) for i, k in enumerate(KERNEL_KINDS)}

    def set_flags(self, flags):
        _check(lib().b2r_set_flags(self._h, flags)); self.flags = flags

    def generate_rays(self, acc):
        out = np.empty((self.width * self.height, 6), np.float32); _check(lib().b2r_generate_rays(self._h, acc, _ptr(out))); return out

    def trace_closest(self, rays):
        r = np.ascontiguousarray(rays, np.float32); n = len(r); t = np.empty(n, np.float32); p = np.empty(n, np.int32)
        _check(lib().b2r_trace_closest(self._h, _ptr(r), n, _ptr(t), _ptr(p))); return t, p

    def trace_shadow(self, rays, tfar):
        r = np.ascontiguousarray(rays, np.float32); tf = np.ascontiguousarray(tfar, np.float32); n = len(r); o = np.empty(n, np.uint8)
        _check(lib().b2r_trace_shadow(self._h, _ptr(r), _ptr(tf), n, _ptr(o))); return o

    def trace_kernel_closest(self, rays, tail=None, origin_prim=None):
        """k_intersect_closest, the per-lane closest-hit kernel of bounces >= 1, on caller rays (b2r_trace_kernel). tail (n bools, with
        FLAG_REFERENCE_EXACT): rays that take the scalar-tail sphere formula. origin_prim (n ints, BVH order; -1 = the root; None = all
        from the root): ray i's walk starts at the node holding that sphere and climbs. Returns (tfar, prim) as trace_closest."""
        r = np.ascontiguousarray(rays, np.float32); n = len(r); t = np.empty(n, np.float32); p = np.empty(n, np.int32)
        tl = None if tail is None else np.ascontiguousarray(tail, np.uint8)
        op = None if origin_prim is None else np.ascontiguousarray(origin_prim, np.int32)
        _check(lib().b2r_trace_kernel(self._h, TAP_CLOSEST, _ptr(r), None, _ptr(op), _ptr(tl), n, 0, _ptr(t), _ptr(p), None)); return t, p

    def trace_kernel_shadow(self, rays, tfar, origin_prim):
        """k_intersect_shadow, the climbing any-hit kernel, on caller rays: ray i's walk starts at the node holding sphere origin_prim[i]
        (BVH order; -1 = the root). Returns occlusion flags as trace_shadow."""
        r = np.ascontiguousarray(rays, np.float32); tf = np.ascontiguousarray(tfar, np.float32); op = np.ascontiguousarray(origin_prim, np.int32)
        n = len(r); o = np.empty(n, np.uint8)
        _check(lib().b2r_trace_kernel(self._h, TAP_SHADOW, _ptr(r), _ptr(tf), _ptr(op), None, n, 0, None, None, _ptr(o))); return o

    def trace_kernel_packet(self, acc):
        """k_intersect_packet, the camera-ray kernel, on the camera rays of sample index acc: (tfar, prim) per pixel in tile order, entry t
        for ray t of generate_rays(acc)."""
        n = self.width * self.height; t = np.empty(n, np.float32); p = np.empty(n, np.int32)
        _check(lib().b2r_trace_kernel(self._h, TAP_PACKET, None, None, None, None, n, acc, _ptr(t), _ptr(p), None)); return t, p

    def link_tables(self):
        """(parent, leaf_node) of the device tree as k_link_tables wrote them (b2r_read_link_tables)."""
        n = C.c_uint32(0); _check(lib().b2r_read_wide_nodes(self._h, None, C.byref(n), None))
        parent = np.empty(n.value, np.uint32); leaf = np.empty(len(self.scene.prims), np.uint32)
        _check(lib().b2r_read_link_tables(self._h, _ptr(parent), _ptr(leaf))); return parent, leaf

    def read_sky_tables(self):
        """B2R_FLAG_SKY_LIGHT: the sky's tables as the device built them (b2r_read_sky_tables): (marginal[H'+1], conditional[H'][W'+1],
        pdf[h][w]), float32."""
        cols = C.c_uint32(0); rows = C.c_uint32(0)
        _check(lib().b2r_read_sky_tables(self._h, None, None, None, C.byref(cols), C.byref(rows)))
        h, w = self.scene.hdri.shape[:2]
        marg = np.empty(rows.value + 1, np.float32); cond = np.empty((rows.value, cols.value + 1), np.float32); pdf = np.empty((h, w), np.float32)
        _check(lib().b2r_read_sky_tables(self._h, _ptr(marg), _ptr(cond), _ptr(pdf), C.byref(cols), C.byref(rows)))
        return marg, cond, pdf

    def read_light_tree(self):
        """B2R_FLAG_LIGHT_TREE: the light tree as the device holds it (b2r_read_light_tree): (nodes[N][8] float32 = {c.xyz, R^2, E, link, 0, 0}
        with link an int32 in the float's bits, light_prim[n_lights] int32 = each light's BVH-order sphere)."""
        n = C.c_uint32(0)
        _check(lib().b2r_read_light_tree(self._h, None, None, C.byref(n)))
        nodes = np.empty((n.value, 8), np.float32); light_prim = np.empty(len(self.scene.lights), np.int32)
        _check(lib().b2r_read_light_tree(self._h, _ptr(nodes), _ptr(light_prim), C.byref(n)))
        return nodes, light_prim

    def wide_nodes(self):
        n = C.c_uint32(0); ms = C.c_uint32(0)
        _check(lib().b2r_read_wide_nodes(self._h, None, C.byref(n), C.byref(ms)))
        out = np.zeros((n.value, 4, 8), np.float32)
        _check(lib().b2r_read_wide_nodes(self._h, _ptr(out), C.byref(n), C.byref(ms)))
        return out, ms.value

    def origin_box(self):
        """{lo.xyz, hi.xyz} the traversal tree's leaf extents were computed for (b2r_get_origin_box)."""
        out = np.zeros(6, np.float32); _check(lib().b2r_get_origin_box(self._h, _ptr(out))); return out


def host_register(arr):
    """Page-lock a numpy frame buffer (what the C++ faces do with their `framebuffer` vector after Resize)."""
    _check(lib().b2r_host_register(_ptr(arr), arr.nbytes))


def host_unregister(arr):
    _check(lib().b2r_host_unregister(_ptr(arr)))


def write_hdr(path, rgba):
    """Image::Store (Image.cpp:71-74): Radiance .hdr of an (H, W, 4) float32 frame, vertically flipped like the reference."""
    a = np.ascontiguousarray(rgba, np.float32)
    _check(lib().b2r_write_hdr(str(path).encode(), _ptr(a), a.shape[1], a.shape[0]))


def read_hdr(path):
    """stbi_loadf(path, &w, &h, &channels, 4) for a Radiance .hdr, as Application.cpp:225-231 loads the sky: (H, W, 4) float32."""
    w, h = C.c_int32(0), C.c_int32(0)
    if lib().b2r_read_hdr(str(path).encode(), None, C.byref(w), C.byref(h)) != OK:
        raise B2RError(ERR_ARG, f"{path}: not a Radiance .hdr stb_image would load")
    out = np.empty((h.value, w.value, 4), np.float32)
    if lib().b2r_read_hdr(str(path).encode(), _ptr(out), C.byref(w), C.byref(h)) != OK:
        raise B2RError(ERR_ARG, f"{path}: corrupt or truncated .hdr")
    return out


def tile_to_raster(buf, width, height):
    """[..., npix] in tile order (t = tile*256 + ID, Renderer.hpp:85-88) -> [..., height, width]."""
    ht, vt = width // 16, height // 16
    a = np.asarray(buf).reshape(buf.shape[:-1] + (vt, ht, 16, 16))
    return np.moveaxis(a, -2, -3).reshape(buf.shape[:-1] + (height, width))
