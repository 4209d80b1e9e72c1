"""CPU oracle for the FSPT hot path -- TEST INFRASTRUCTURE, never imported by fspt_b200/.

ctypes front-end of oracle/libfspt_oracle.so (sources: fspt_oracle.cpp, fspt_oracle_host.cpp,
oracle_math.h, oracle_texunit.h; recipe: oracle/Makefile).  The shader restatement is pinned bit for bit to the
reference's own shader sources executed on the CPU (oracle/reference_shaders.py, tests/test_reference_pin.py); see the
header of fspt_oracle.cpp for what that covers.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libfspt_oracle.so")


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("fspt_oracle.cpp", "fspt_oracle_host.cpp", "oracle_math.h", "oracle_texunit.h", "Makefile")]
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs if os.path.exists(s)):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB


class OScene(C.Structure):
    _fields_ = [
        ("bvh", C.c_void_p), ("tris", C.c_void_p), ("mats", C.c_void_p), ("norms", C.c_void_p),
        ("uvs", C.c_void_p), ("atlas", C.c_void_p), ("env", C.c_void_p), ("bins", C.c_void_p),
        ("n_nodes", C.c_int32), ("n_tris", C.c_int32), ("atlas_res", C.c_int32), ("atlas_layers", C.c_int32),
        ("env_w", C.c_int32), ("env_h", C.c_int32), ("n_bins", C.c_int32), ("leaf_size", C.c_int32),
    ]


class OStats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("node_visits", C.c_uint64), ("leaf_visits", C.c_uint64),
                ("stack_overflow", C.c_uint64), ("capped", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.oracle_bvh_build.restype = C.c_int
        _lib.oracle_bvh_build2.restype = C.c_int
        _lib.oracle_env_bins.restype = C.c_int
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class Oracle:
    """Holds one scene in the reference's flattened layout (SURVEY.md App. A)."""

    def __init__(self, arrays, leaf_size=4):
        # arrays: any object with bvh/tris/mats/norms/uvs/atlas/env/bins numpy attributes
        self.bvh = _f32(arrays.bvh).reshape(-1, 9)
        self.tris = _f32(arrays.tris).reshape(-1, 9)
        self.mats = _f32(arrays.mats).reshape(-1, 12)
        self.norms = _f32(arrays.norms).reshape(-1, 27)
        self.uvs = _f32(arrays.uvs).reshape(-1, 6)
        self.atlas = np.ascontiguousarray(arrays.atlas, dtype=np.uint8)
        self.env = np.ascontiguousarray(arrays.env, dtype=np.uint8)
        self.bins = np.ascontiguousarray(arrays.bins, dtype=np.uint16).reshape(-1, 4)
        assert self.atlas.ndim == 4 and self.atlas.shape[1] == self.atlas.shape[2] and self.atlas.shape[3] == 4
        assert self.env.ndim == 3 and self.env.shape[2] == 4
        s = OScene()
        s.bvh, s.tris, s.mats, s.norms, s.uvs = _p(self.bvh), _p(self.tris), _p(self.mats), _p(self.norms), _p(self.uvs)
        s.atlas, s.env, s.bins = _p(self.atlas), _p(self.env), _p(self.bins)
        s.n_nodes, s.n_tris = self.bvh.shape[0], self.tris.shape[0]
        s.atlas_layers, s.atlas_res = self.atlas.shape[0], self.atlas.shape[1]
        s.env_h, s.env_w = self.env.shape[0], self.env.shape[1]
        s.n_bins, s.leaf_size = self.bins.shape[0], leaf_size
        self.s = s

    def bvh_test(self, pos4, dir4, nthreads=0, anyhit=False):
        """(index, t, count, stats) of intersectScene per ray; anyhit: stop after the first leaf that yields a hit, as the
        product's hit-or-miss rays do (FSPT_PARAM_ANYHIT)"""
        pos4, dir4 = _f32(pos4).reshape(-1, 4), _f32(dir4).reshape(-1, 4)
        n = pos4.shape[0]
        idx = np.empty(n, np.int32); t = np.empty(n, np.float32); cnt = np.empty(n, np.int32)
        st = OStats()
        lib().oracle_bvh_test(C.byref(self.s), _p(pos4), _p(dir4), C.c_int(n), _p(idx), _p(t), _p(cnt), C.byref(st),
                              C.c_int(nthreads), C.c_int(1 if anyhit else 0))
        return idx, t, cnt, st.as_dict()

    def brute_force(self, pos4, dir4, nthreads=0):
        pos4, dir4 = _f32(pos4).reshape(-1, 4), _f32(dir4).reshape(-1, 4)
        n = pos4.shape[0]
        idx = np.empty(n, np.int32); t = np.empty(n, np.float32)
        lib().oracle_brute_force(C.byref(self.s), _p(pos4), _p(dir4), C.c_int(n), _p(idx), _p(t), C.c_int(nthreads))
        return idx, t

    def trace(self, pos4, dir4, W, H, tick, rand_base, env_theta, fb_prev=None, sanitize=1, max_refractions=64,
              nthreads=0, want_color=False):
        pos4, dir4 = _f32(pos4).reshape(-1, 4), _f32(dir4).reshape(-1, 4)
        assert pos4.shape[0] == W * H
        fb_prev = _f32(fb_prev).reshape(-1, 4) if fb_prev is not None else None
        out = np.empty((H, W, 4), np.float32)
        col = np.empty((H, W, 4), np.float32) if want_color else None
        st = OStats()
        lib().oracle_trace(C.byref(self.s), _p(pos4), _p(dir4), C.c_int(W), C.c_int(H), C.c_uint32(tick),
                           C.c_float(rand_base), C.c_float(env_theta), _p(fb_prev), _p(out), _p(col),
                           C.c_int(sanitize), C.c_int(max_refractions), C.byref(st), C.c_int(nthreads))
        return (out, col, st.as_dict()) if want_color else (out, st.as_dict())


def camera(W, H, P, I, fov_scale, lens, rand_base, nthreads=0):
    P, I, lens = _f32(P), _f32(I), _f32(lens)
    pos = np.empty((H, W, 4), np.float32); d = np.empty((H, W, 4), np.float32)
    lib().oracle_camera(C.c_int(W), C.c_int(H), _p(P), _p(I), C.c_float(fov_scale), _p(lens), C.c_float(rand_base),
                        _p(pos), _p(d), C.c_int(nthreads))
    return pos, d


def draw(fb, exposure=1.0, saturation=1.0, denoise=False, max_sigma=2.0, scale=1.0, nthreads=0):
    fb = _f32(fb)
    H, W = fb.shape[0], fb.shape[1]
    out = np.empty((H, W, 4), np.uint8)
    lib().oracle_draw(_p(fb), C.c_int(W), C.c_int(H), C.c_float(exposure), C.c_float(saturation),
                      C.c_int(1 if denoise else 0), C.c_float(max_sigma), C.c_float(scale), _p(out), C.c_int(nthreads))
    return out


# the probe codes of fspt_debug_math (include/fspt_b200.h), answered with the model's plain operations
DM_CODES = {"sin": 0, "cos": 1, "atan2": 2, "asin": 3, "exp2": 4, "pow": 5, "sincos_s": 6, "sincos_c": 7, "log2": 8,
            "rnd": 9, "min": 10, "max": 11, "clamp": 12, "div": 13, "div_shared": 14, "div_z": 15, "coord_to_i32": 16,
            "quant8": 17}
# the packed f32x2 lanes of the slab test, answered with the scalar IEEE operation
DM_PACKED_CODES = {"sub2_lo": 32, "sub2_hi": 33, "mul2_lo": 34, "mul2_hi": 35}


def dm_eval(fn, x, y=None):
    x = _f32(x).ravel(); y = _f32(y).ravel() if y is not None else np.zeros_like(x)
    out = np.empty_like(x)
    code = DM_CODES[fn] if fn in DM_CODES else DM_PACKED_CODES[fn]
    if lib().oracle_dm_eval(C.c_int(code), _p(x), _p(y), _p(out), C.c_int(x.size)) != 0:
        raise ValueError("oracle_dm_eval: unknown probe %r" % (fn,))
    return out


def bvh_build(verts, max_tris=4, box_verts=None):
    """bvh.js + main.js flatten.  verts: (T,3,3) float64.  Returns (nodes[N,9] f32 masked, order[T] i32, depth)."""
    verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 9)
    if box_verts is not None:
        box_verts = np.ascontiguousarray(box_verts, dtype=np.float64).reshape(-1, 9)
    T = verts.shape[0]
    nodes = np.empty((2 * T + 1, 9), np.float32); order = np.empty(T, np.int32); depth = C.c_int32(0)
    n = lib().oracle_bvh_build2(_p(verts), _p(box_verts), C.c_int(T), C.c_int(max_tris), _p(nodes), _p(order), C.byref(depth))
    if n < 0:
        raise RuntimeError("bvh.js would crash / recurse forever on this input")
    return nodes[:n].copy(), order, int(depth.value)


def env_bins(rgba8):
    rgba8 = np.ascontiguousarray(rgba8, dtype=np.uint8)
    H, W = rgba8.shape[0], rgba8.shape[1]
    cap = 4 * 65536
    out = np.empty(cap, np.uint16)
    n = lib().oracle_env_bins(_p(rgba8), C.c_int(W), C.c_int(H), _p(out), C.c_int(cap))
    return out[:n].reshape(-1, 4).copy()


def pack_layer(pixels, res, corrected=False, swizzle=None):
    """texture_packer.js blit, literal per-fragment restatement."""
    pixels = np.ascontiguousarray(pixels, dtype=np.uint8)
    h, w = pixels.shape[0], pixels.shape[1]
    out = np.empty((res, res, 4), np.uint8)
    sw = np.asarray(swizzle, np.int32) if swizzle is not None else None
    lib().oracle_pack_layer(_p(pixels), C.c_int(w), C.c_int(h), C.c_int(res), C.c_int(1 if corrected else 0), _p(sw), _p(out))
    return out
