"""ctypes binding of libfspt_b200.so (include/fspt_b200.h).  Plumbing only: every compute call goes to the
CUDA library; there is no Python/CPU fallback (calls raise FsptError when the library or a B200 is missing)."""
import ctypes as C
import os

import numpy as np

from . import build as _build

FSPT_OK = 0


class FsptError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("fspt error %d: %s" % (code, msg))
        self.code = code


class SceneDesc(C.Structure):
    _fields_ = [
        ("bvh", C.c_void_p), ("triangles", C.c_void_p), ("materials", C.c_void_p), ("normals", C.c_void_p),
        ("uvs", C.c_void_p), ("lights", C.c_void_p), ("light_ranges", C.c_void_p), ("atlas", C.c_void_p),
        ("env", C.c_void_p), ("radiance_bins", C.c_void_p),
        ("n_nodes", C.c_int32), ("n_triangles", C.c_int32), ("n_light_triangles", C.c_int32),
        ("n_light_ranges", C.c_int32), ("atlas_res", C.c_int32), ("atlas_layers", C.c_int32),
        ("env_width", C.c_int32), ("env_height", C.c_int32), ("env_bins", C.c_int32), ("leaf_size", C.c_int32),
    ]


class FrameParams(C.Structure):
    _fields_ = [("eye", C.c_float * 3), ("dir", C.c_float * 3), ("fov_scale", C.c_float),
                ("lens_features", C.c_float * 2), ("env_theta", C.c_float)]


class PostParams(C.Structure):
    _fields_ = [("exposure", C.c_float), ("saturation", C.c_float), ("max_sigma", C.c_float), ("scale", C.c_float),
                ("denoise", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("rays", C.c_uint64), ("node_visits", C.c_uint64), ("leaf_visits", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("trace_ms", C.c_double), ("render_ms", C.c_double),
                ("last_rays", C.c_uint64), ("last_node_visits", C.c_uint64), ("last_leaf_visits", C.c_uint64),
                ("capped_paths", C.c_uint64), ("shade_ms", C.c_double), ("reduce_ms", C.c_double),
                ("primary_trace_ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


EXPORTS = [
    "fspt_abi_version", "fspt_create", "fspt_destroy", "fspt_last_error", "fspt_scene_upload", "fspt_clear",
    "fspt_render", "fspt_resolve", "fspt_read_accum", "fspt_write_accum", "fspt_set_accum_mode",
    "fspt_accum_device_ptr", "fspt_set_accum_samples", "fspt_debug_primary", "fspt_debug_trace",
    "fspt_debug_last_color", "fspt_debug_math", "fspt_debug_read_bandwidth", "fspt_get_stats", "fspt_synchronize", "fspt_bvh_build", "fspt_bvh_build2",
    "fspt_env_bins", "fspt_pack_layer", "fspt_set_param", "fspt_set_tile", "fspt_comm_unique_id", "fspt_comm_init",
    "fspt_comm_destroy", "fspt_reduce_accum", "fspt_scene_broadcast", "fspt_scene_upload_async", "fspt_scene_upload_wait",
    "fspt_host_register", "fspt_host_unregister", "fspt_debug_pack_scene", "fspt_bvh_build_device", "fspt_device_check",
    "fspt_set_adaptive", "fspt_active_pixels", "fspt_read_moment", "fspt_write_moment",
]
PARAM_ANYHIT, PARAM_MAX_REFRACTIONS, PARAM_SANITIZE_NAN = 1, 2, 3

_lib = None


def lib_path():
    return _build.LIB


def load(build_if_needed=True):
    """Load the shared library (building it in-tree first if sources are newer).  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("FSPT_LIB") or _build.LIB  # FSPT_LIB: A/B kernel variants (tools/quick.py)
    if path == _build.LIB and build_if_needed and os.path.exists(_build.NVCC):
        _build.build()
    if not os.path.exists(path):
        raise FsptError(-2, "%s is not built (run `python -m fspt_b200.build`); there is no CPU fallback" % path)
    lib = C.CDLL(path)
    lib.fspt_last_error.restype = C.c_char_p
    lib.fspt_last_error.argtypes = [C.c_void_p]
    lib.fspt_destroy.restype = None
    lib.fspt_destroy.argtypes = [C.c_void_p]
    for name in EXPORTS:
        try:
            getattr(lib, name)  # AttributeError here = header and library disagree
        except AttributeError:
            if not os.environ.get("FSPT_LIB"):  # an explicitly chosen A/B variant may predate an entry point
                raise
    _lib = lib
    return lib


def comm_unique_id():
    """fspt_comm_unique_id: 128 bytes from ncclGetUniqueId (rank 0 calls it, the host ships it to the other ranks)."""
    lib = load()
    buf = (C.c_uint8 * 128)()
    rc = lib.fspt_comm_unique_id(buf)
    if rc != FSPT_OK:
        raise FsptError(rc, (lib.fspt_last_error(None) or b"").decode())
    return bytes(buf)


def host_register(a):
    """fspt_host_register: page-lock a C-contiguous numpy array in place (uploads then DMA it from where it lies)."""
    lib = load()
    assert a.flags["C_CONTIGUOUS"]
    rc = lib.fspt_host_register(a.ctypes.data_as(C.c_void_p), C.c_uint64(a.nbytes))
    if rc != FSPT_OK:
        raise FsptError(rc, (lib.fspt_last_error(None) or b"").decode())
    return a


def host_unregister(a):
    lib = load()
    rc = lib.fspt_host_unregister(a.ctypes.data_as(C.c_void_p))
    if rc != FSPT_OK:
        raise FsptError(rc, (lib.fspt_last_error(None) or b"").decode())


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def bvh_build(verts, max_tris=4, n_threads=0, box_verts=None):
    """fspt_bvh_build(2): bvh.js + serializeTree + flatten.  Returns (nodes[N,9] f32 masked, order[T] i32, depth).
    box_verts: vertices the stale Triangle.boundingBox was computed from (scene.normalize), default = verts."""
    lib = load()
    verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 9)
    T = verts.shape[0]
    if box_verts is not None:
        box_verts = np.ascontiguousarray(box_verts, dtype=np.float64).reshape(-1, 9)
        assert box_verts.shape == verts.shape
    nodes = np.empty((2 * T + 1, 9), np.float32)
    order = np.empty(T, np.int32)
    n = C.c_int32(0)
    depth = C.c_int32(0)
    rc = lib.fspt_bvh_build2(ptr(verts), ptr(box_verts), C.c_int32(T), C.c_int32(max_tris), ptr(nodes), ptr(order),
                             C.byref(n), C.byref(depth), C.c_int32(n_threads))
    if rc != FSPT_OK:
        raise FsptError(rc, "fspt_bvh_build failed (degenerate input: the JavaScript builder would not terminate)")
    return nodes[: n.value].copy(), order, int(depth.value)


def bvh_build_device(verts, max_tris=4, box_verts=None, device=0):
    """fspt_bvh_build_device: the same tree as bvh_build, built on CUDA device `device`.  Returns (nodes, order, depth)."""
    lib = load()
    verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 9)
    T = verts.shape[0]
    if box_verts is not None:
        box_verts = np.ascontiguousarray(box_verts, dtype=np.float64).reshape(-1, 9)
        assert box_verts.shape == verts.shape
    nodes = np.empty((2 * T + 1, 9), np.float32)
    order = np.empty(T, np.int32)
    n = C.c_int32(0)
    depth = C.c_int32(0)
    rc = lib.fspt_bvh_build_device(C.c_int32(device), ptr(verts), ptr(box_verts), C.c_int32(T), C.c_int32(max_tris),
                                   ptr(nodes), ptr(order), C.byref(n), C.byref(depth))
    if rc != FSPT_OK:
        raise FsptError(rc, (lib.fspt_last_error(None) or b"").decode())
    return nodes[: n.value].copy(), order, int(depth.value)


def device_usable(device=0):
    """fspt_device_check: True when CUDA device `device` is an sm_100 device the library's kernels run on."""
    return load().fspt_device_check(C.c_int32(device)) == FSPT_OK


def env_bins(rgba8):
    """fspt_env_bins: ProcessEnvRadiance.  rgba8 (H,W,4) uint8 RGBE.  Returns (B,4) uint16."""
    lib = load()
    rgba8 = np.ascontiguousarray(rgba8, dtype=np.uint8)
    H, W = rgba8.shape[0], rgba8.shape[1]
    cap = 4 * 65536
    out = np.empty(cap, np.uint16)
    n = C.c_int32(0)
    rc = lib.fspt_env_bins(ptr(rgba8), C.c_int32(W), C.c_int32(H), ptr(out), C.c_int32(cap), C.byref(n))
    if rc != FSPT_OK:
        raise FsptError(rc, "fspt_env_bins failed")
    return out[: n.value].reshape(-1, 4).copy()


def pack_layer(pixels, res, corrected=False, swizzle=None, n_threads=0):
    """fspt_pack_layer: one image layer of the atlas.  pixels (h,w,4) uint8, row 0 = image top -> (res,res,4) uint8."""
    lib = load()
    pixels = np.ascontiguousarray(pixels, dtype=np.uint8)
    h, w = pixels.shape[0], pixels.shape[1]
    out = np.empty((res, res, 4), np.uint8)
    sw = np.asarray(swizzle, np.int32) if swizzle is not None else None
    rc = lib.fspt_pack_layer(ptr(pixels), C.c_int32(w), C.c_int32(h), C.c_int32(res), C.c_int32(1 if corrected else 0),
                             ptr(sw), ptr(out), C.c_int32(n_threads))
    if rc != FSPT_OK:
        raise FsptError(rc, "fspt_pack_layer failed (bad size or swizzle)")
    return out


def scene_desc(sa, keep):
    """fspt_scene_desc over the arrays of a SceneArrays-like object; `keep` receives the (possibly converted) arrays the
    pointers refer to and must outlive the call that uses the descriptor."""
    d = SceneDesc()
    keep.update(
        bvh=f32(sa.bvh), tris=f32(sa.tris), mats=f32(sa.mats), norms=f32(sa.norms), uvs=f32(sa.uvs),
        atlas=np.ascontiguousarray(sa.atlas, np.uint8), env=np.ascontiguousarray(sa.env, np.uint8),
        bins=np.ascontiguousarray(sa.bins, np.uint16))
    lights = getattr(sa, "lights", None)
    ranges = getattr(sa, "light_ranges", None)
    if lights is not None and len(lights):
        keep["lights"] = f32(lights)
        keep["ranges"] = f32(ranges)
        d.lights, d.light_ranges = ptr(keep["lights"]), ptr(keep["ranges"])
        d.n_light_triangles = keep["lights"].size // 9
        d.n_light_ranges = keep["ranges"].size // 2
    d.bvh, d.triangles, d.materials = ptr(keep["bvh"]), ptr(keep["tris"]), ptr(keep["mats"])
    d.normals, d.uvs, d.atlas, d.env = ptr(keep["norms"]), ptr(keep["uvs"]), ptr(keep["atlas"]), ptr(keep["env"])
    d.radiance_bins = ptr(keep["bins"])
    d.n_nodes = keep["bvh"].size // 9
    d.n_triangles = keep["tris"].size // 9
    d.atlas_layers, d.atlas_res = keep["atlas"].shape[0], keep["atlas"].shape[1]
    d.env_height, d.env_width = keep["env"].shape[0], keep["env"].shape[1]
    d.env_bins = keep["bins"].size // 4
    d.leaf_size = getattr(sa, "leaf_size", 4)
    return d


def debug_pack_scene(sa, n_threads=0):
    """fspt_debug_pack_scene: the host half of fspt_scene_upload, no GPU.  Returns a dict with node64 (NI,16) f32,
    tri48 (T+3,12) f32, shaderec (T,48) f32, mat_id (T,) i32 and the info fields."""
    lib = load()
    keep = {}
    d = scene_desc(sa, keep)
    info = np.zeros(5, np.int32)

    def ck(rc):
        if rc != FSPT_OK:
            raise FsptError(rc, (lib.fspt_last_error(None) or b"").decode())
    ck(lib.fspt_debug_pack_scene(C.byref(d), None, None, None, None, ptr(info), C.c_int32(n_threads)))
    ni, T = int(info[0]), d.n_triangles
    node64 = np.zeros((max(ni, 1), 16), np.float32)
    tri48 = np.zeros((T + 3, 12), np.float32)
    shaderec = np.zeros((T, 48), np.float32)
    mat_id = np.zeros(T, np.int32)
    ck(lib.fspt_debug_pack_scene(C.byref(d), ptr(node64), ptr(tri48), ptr(shaderec), ptr(mat_id), ptr(info), C.c_int32(n_threads)))
    return dict(node64=node64[:ni] if ni else node64, tri48=tri48, shaderec=shaderec, mat_id=mat_id, n_interior=ni,
                n_materials=int(info[1]), root_ref=int(info[2]), dielectric=bool(info[3]), depth=int(info[4]))


class Context:
    """Thin RAII wrapper over fspt_ctx."""

    def __init__(self, width, height, device=0):
        self.lib = load()
        self.h = C.c_void_p()
        self.width, self.height = int(width), int(height)
        rc = self.lib.fspt_create(C.byref(self.h), C.c_int32(width), C.c_int32(height), C.c_int32(device))
        if rc != FSPT_OK:
            raise FsptError(rc, (self.lib.fspt_last_error(None) or b"").decode())
        self._keep = None

    def _ck(self, rc):
        if rc != FSPT_OK:
            raise FsptError(rc, (self.lib.fspt_last_error(self.h) or b"").decode())

    def close(self):
        if self.h:
            self.lib.fspt_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def scene_upload(self, sa, wait=True):
        """fspt_scene_upload; wait=False: fspt_scene_upload_async -- returns once everything but the atlas has been
        consumed, the atlas is staged in the background (the arrays are kept alive here until upload_wait / the next
        upload) and the next render's primary traversal overlaps it."""
        keep = {}
        d = scene_desc(sa, keep)
        if wait:
            self._ck(self.lib.fspt_scene_upload(self.h, C.byref(d)))
            self._keep = None
        else:
            self._keep = None  # (the library joins the previous staging thread before it touches anything)
            self._ck(self.lib.fspt_scene_upload_async(self.h, C.byref(d)))
            self._keep = keep
        return sum(v.nbytes for v in keep.values())

    def upload_wait(self):
        """fspt_scene_upload_wait: the atlas of the last asynchronous upload has been staged; its buffers are released."""
        try:
            self._ck(self.lib.fspt_scene_upload_wait(self.h))
        finally:
            self._keep = None

    @staticmethod
    def frame(eye, dir_, fov_scale, lens_features, env_theta):
        f = FrameParams()
        f.eye[:] = [float(x) for x in eye]
        f.dir[:] = [float(x) for x in dir_]
        f.fov_scale = float(fov_scale)
        f.lens_features[:] = [float(x) for x in lens_features]
        f.env_theta = float(env_theta)
        return f

    def set_param(self, key, value):
        self._ck(self.lib.fspt_set_param(self.h, C.c_int32(key), C.c_int32(value)))

    def clear(self):
        self._ck(self.lib.fspt_clear(self.h))

    def render(self, frame, first_tick, rand_base_camera, rand_base_tracer):
        rc_, rt_ = f32(rand_base_camera).ravel(), f32(rand_base_tracer).ravel()
        assert rc_.size == rt_.size
        self._ck(self.lib.fspt_render(self.h, C.byref(frame), C.c_uint32(first_tick), C.c_int32(rc_.size), ptr(rc_), ptr(rt_)))

    def synchronize(self):
        self._ck(self.lib.fspt_synchronize(self.h))

    def resolve(self, exposure=1.0, saturation=1.0, denoise=False, max_sigma=2.0, scale=1.0, out=None):
        p = PostParams(float(exposure), float(saturation), float(max_sigma), float(scale), 1 if denoise else 0)
        if out is None:
            out = np.empty((self.height, self.width, 4), np.uint8)
        self._ck(self.lib.fspt_resolve(self.h, C.byref(p), ptr(out)))
        return out

    def read_accum(self):
        out = np.empty((self.height, self.width, 4), np.float32)
        self._ck(self.lib.fspt_read_accum(self.h, ptr(out)))
        return out

    def write_accum(self, fb, next_tick):
        fb = f32(fb)
        assert fb.size == self.width * self.height * 4
        self._ck(self.lib.fspt_write_accum(self.h, ptr(fb), C.c_uint32(next_tick)))

    def set_accum_mode(self, mode):
        self._ck(self.lib.fspt_set_accum_mode(self.h, C.c_int32(mode)))

    def accum_device_ptr(self):
        p = C.c_void_p()
        n = C.c_uint64(0)
        s = C.c_uint64(0)
        self._ck(self.lib.fspt_accum_device_ptr(self.h, C.byref(p), C.byref(n), C.byref(s)))
        return p.value, int(n.value), int(s.value)

    def set_adaptive(self, max_rel_error, min_samples=16):
        """fspt_set_adaptive: max_rel_error > 0 renders, before each wave, only the pixels whose relative standard error
        of the mean luminance is still above it (or that have fewer than min_samples samples); 0 turns it off.  Sum mode
        only (set_accum_mode(1))."""
        self._ck(self.lib.fspt_set_adaptive(self.h, C.c_float(max_rel_error), C.c_int32(min_samples)))

    def active_pixels(self):
        """fspt_active_pixels: how many pixels of the rectangle the next wave would render (synchronises)."""
        n = C.c_uint64(0)
        self._ck(self.lib.fspt_active_pixels(self.h, C.byref(n)))
        return int(n.value)

    def read_moment(self):
        """fspt_read_moment: per pixel, the f32 sum of the squared luminances of its samples (height, width)."""
        out = np.empty((self.height, self.width), np.float32)
        self._ck(self.lib.fspt_read_moment(self.h, ptr(out)))
        return out

    def write_moment(self, m2):
        m2 = f32(m2)
        assert m2.size == self.width * self.height
        self._ck(self.lib.fspt_write_moment(self.h, ptr(m2)))

    def set_tile(self, x0, y0, w, h):
        """The pixel rectangle of the frame this context renders (GL row order); default = whole frame."""
        self._ck(self.lib.fspt_set_tile(self.h, C.c_int32(x0), C.c_int32(y0), C.c_int32(w), C.c_int32(h)))

    def comm_init(self, unique_id, rank, world):
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        self._ck(self.lib.fspt_comm_init(self.h, buf, C.c_int32(rank), C.c_int32(world)))

    def comm_destroy(self):
        self._ck(self.lib.fspt_comm_destroy(self.h))

    def reduce_accum(self, root=0):
        self._ck(self.lib.fspt_reduce_accum(self.h, C.c_int32(root)))

    def scene_broadcast(self, root=0):
        self._ck(self.lib.fspt_scene_broadcast(self.h, C.c_int32(root)))

    def set_accum_samples(self, n):
        self._ck(self.lib.fspt_set_accum_samples(self.h, C.c_uint64(n)))

    def debug_primary(self, frame, rand_base_camera, want_rays=True):
        P = self.width * self.height
        idx = np.empty(P, np.int32)
        t = np.empty(P, np.float32)
        cnt = np.empty(P, np.int32)
        pos = np.empty((self.height, self.width, 4), np.float32) if want_rays else None
        d = np.empty((self.height, self.width, 4), np.float32) if want_rays else None
        self._ck(self.lib.fspt_debug_primary(self.h, C.byref(frame), C.c_float(rand_base_camera), ptr(idx), ptr(t),
                                             ptr(cnt), ptr(pos), ptr(d)))
        return idx, t, cnt, pos, d

    def debug_trace(self, pos4, dir4):
        pos4, dir4 = f32(pos4).reshape(-1, 4), f32(dir4).reshape(-1, 4)
        n = pos4.shape[0]
        idx = np.empty(n, np.int32)
        t = np.empty(n, np.float32)
        cnt = np.empty(n, np.int32)
        self._ck(self.lib.fspt_debug_trace(self.h, ptr(pos4), ptr(dir4), C.c_int32(n), ptr(idx), ptr(t), ptr(cnt)))
        return idx, t, cnt

    def debug_last_color(self):
        out = np.empty((self.height, self.width, 4), np.float32)
        self._ck(self.lib.fspt_debug_last_color(self.h, ptr(out)))
        return out

    def debug_read_bandwidth(self, nbytes, iters=20):
        """GB/s of a streaming read over an nbytes buffer (L2 ceiling when it fits L2, HBM ceiling when it does not)."""
        out = C.c_double(0.0)
        self._ck(self.lib.fspt_debug_read_bandwidth(self.h, C.c_uint64(int(nbytes)), C.c_int32(int(iters)), C.byref(out)))
        return out.value

    def debug_math(self, fn, x, y=None):
        names = {"sin": 0, "cos": 1, "atan2": 2, "asin": 3, "exp2": 4, "pow": 5, "sincos_s": 6, "sincos_c": 7}
        x = f32(x).ravel()
        y = f32(y).ravel() if y is not None else None
        out = np.empty_like(x)
        self._ck(self.lib.fspt_debug_math(self.h, C.c_int32(names[fn]), ptr(x), ptr(y), ptr(out), C.c_int32(x.size)))
        return out

    def stats(self):
        s = Stats()
        self._ck(self.lib.fspt_get_stats(self.h, C.byref(s)))
        return s.as_dict()
