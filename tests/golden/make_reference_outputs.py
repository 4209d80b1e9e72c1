#!/usr/bin/env python
"""Records tests/golden/reference_shaders/outputs.npz: what the reference's OWN fragment shaders (camera.fs, bvh_test.fs,
tracer.fs, draw.fs, compiled for the CPU by `make -C oracle ref`, oracle/reference_shaders.py) compute on the inputs of
tests/test_reference_pin.py and of tests/test_gpu_parity.py::test_cuda_against_the_reference_shaders_themselves.
Those tests compare the oracle restatement and the CUDA path with these records, so they run wherever the repository
is, without the reference tree or a compiler for its shaders.

Each output is stored as a SHA-256 digest of its bits (every NaN counted as one value, as the tests' bit comparison
does) and a fixed sample of its values: the digest makes the comparison as strict as one against the whole array, the
sample says where a mismatch lies.  The oracle restatement must give the same bits as the shaders (asserted below
before anything is written).
    python tests/golden/make_reference_outputs.py
"""
import hashlib
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "reference_shaders", "outputs.npz")  # apart from the scene fixtures of test_golden.py
N_SAMPLE = 64

_stores = {}


def canonical(a):
    """The bits the tests compare: float32 as uint32 with every NaN one pattern (NaN payloads are not compared)."""
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        b = a.view(np.uint32).copy()
        b[np.isnan(a)] = 0x7FC00000
        return b
    return a


def digest(a):
    c = canonical(a)
    h = hashlib.sha256(("%s %s\n" % (c.dtype.str, c.shape)).encode())
    h.update(c.tobytes())
    return h.hexdigest()


def record(out, key, a):
    a = np.ascontiguousarray(a)
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    idx = np.sort(rng.choice(a.size, min(a.size, N_SAMPLE), replace=False)).astype(np.int64)
    out[key + ":sha256"] = np.array(digest(a))
    out[key + ":shape"] = np.array(a.shape, np.int64)
    out[key + ":idx"] = idx
    out[key + ":val"] = a.reshape(-1)[idx]


def check(key, got, path=PATH):
    """Asserts that `got` has the bits the reference's shaders computed for `key` (stored in `path`)."""
    if path not in _stores:
        with np.load(path) as z:
            _stores[path] = {k: z[k] for k in z.files}
    _store = _stores[path]
    got = np.ascontiguousarray(got)
    shape = tuple(int(x) for x in _store[key + ":shape"])
    assert got.shape == shape, "%s: shape %s, the reference's is %s" % (key, got.shape, shape)
    idx, val = _store[key + ":idx"], _store[key + ":val"]
    sample = got.reshape(-1)[idx]
    bad = np.flatnonzero(canonical(sample) != canonical(val))
    assert bad.size == 0, "%s: %d of %d sampled values differ from the reference's; first at flat index %d: %r, reference %r" % (
        key, bad.size, idx.size, idx[bad[0]], sample[bad[0]], val[bad[0]])
    assert digest(got) == str(_store[key + ":sha256"]), \
        "%s: differs from the reference's output (its %d sampled values agree)" % (key, idx.size)


def beq(a, b):
    return np.array_equal(canonical(a), canonical(b))


def make_pin(out, oracle, R):
    """The inputs and calls of tests/test_reference_pin.py, with the reference's shaders in place of the oracle."""
    import test_reference_pin as T
    from fspt_b200 import scenes
    for name, case in zip(T.CAMERA_IDS, T.CAMERAS):
        W, H, P, I, fov, lens, rb = case
        pos, d = R.camera(W, H, P, I, fov, np.asarray(lens, np.float32), rb)
        po, do = oracle.camera(W, H, P, I, fov, np.asarray(lens, np.float32), rb)
        assert beq(pos, po) and beq(d, do), name
        record(out, "camera/%s/pos" % name, pos)
        record(out, "camera/%s/dir" % name, d)
    cam = scenes.BUNNY_CAMERA
    lens = np.asarray(scenes.lens_features(cam), np.float32)
    pos, d = R.camera(3840, 2160, cam["eye"], cam["dir"], cam["fov_scale"], lens, 8191.25)
    po, do = oracle.camera(3840, 2160, cam["eye"], cam["dir"], cam["fov_scale"], lens, 8191.25)
    assert beq(pos, po) and beq(d, do)
    record(out, "camera/3840x2160/pos", pos)
    record(out, "camera/3840x2160/dir", d)

    for name in T.SCENES:
        sa, cam = T.SCENES[name]()
        O, Rf = oracle.Oracle(sa), R.Reference(sa)
        for rays, (p4, d4) in zip(("primary", "random"), T._bvh_rays(oracle, sa, cam)):
            i, t, c, heat = Rf.bvh_test(p4, d4, want_heat=True)
            io, to, co, _ = O.bvh_test(p4, d4)
            assert beq(i, io) and beq(t, to) and beq(c, co), name
            for what, a in (("index", i), ("t", t), ("count", c), ("heat", heat[:, 0])):
                record(out, "bvh_test/%s/%s/%s" % (name, rays, what), a)

    for name, W, H, ticks in T.TRACER_CASES:
        sa, cam = T.SCENES[name]()
        O, Rf = oracle.Oracle(sa), R.Reference(sa)
        rc, rt = scenes.rand_bases(ticks, 41)
        fr = fo = None
        for k in range(ticks):
            pos, d = T._primary(oracle, sa, cam, W, H, rc[k])
            fr = Rf.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fr)
            fo, _ = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fo, sanitize=0, max_refractions=1 << 20)
            assert beq(fr, fo), (name, k)
            record(out, "tracer/%s/tick%d" % (name, k), fr)

    sa, cam = T.SCENES["bunny"]()
    O, Rf = oracle.Oracle(sa), R.Reference(sa)
    for theta in T.THETAS:
        pos, d = T._primary(oracle, sa, cam, 48, 32, 3.5)
        fr = Rf.trace(pos, d, 48, 32, 0, 4242.0, theta)
        assert beq(fr, O.trace(pos, d, 48, 32, 0, 4242.0, theta, sanitize=0)[0])
        record(out, "tracer/bunny/theta%r" % theta, fr)

    fb = T._draw_input(oracle)
    for name, post in zip(T.POST_IDS, T.POSTS):
        rgba = R.draw(fb, **post)
        assert beq(rgba, oracle.draw(fb, **post)), name
        record(out, "draw/%s" % name, rgba)


def make_cuda(out, oracle, R):
    """The inputs and calls of test_cuda_against_the_reference_shaders_themselves (tests/test_gpu_parity.py)."""
    import test_gpu_parity as G
    from fspt_b200 import scenes
    sa, cam = scenes.bunny_class(subdiv=4, atlas_res=64, env_size=(256, 128))   # the `small_bunny` fixture
    W, H, N = G.REF_W, G.REF_H, G.REF_N
    Rf = R.Reference(sa)
    lens = np.asarray(scenes.lens_features(cam), np.float32)
    rc, rt = scenes.rand_bases(N, 29)
    pos, d = R.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rc[0])
    record(out, "cuda/camera/pos", pos)
    record(out, "cuda/camera/dir", d)
    i, t, c = Rf.bvh_test(pos, d)
    for what, a in (("index", i), ("t", t), ("count", c)):
        record(out, "cuda/bvh_test/" + what, a)
    fb = None
    for k in range(N):
        p4, d4 = R.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rc[k])
        fb = Rf.trace(p4, d4, W, H, k, rt[k], cam["env_theta"], fb_prev=fb)
    record(out, "cuda/tracer/accum_rgb", fb[..., :3])
    record(out, "cuda/draw/rgba8", R.draw(fb, **G.REF_POST))
    O = oracle.Oracle(sa)
    fo = None
    for k in range(N):
        p4, d4 = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rc[k])
        fo, _ = O.trace(p4, d4, W, H, k, rt[k], cam["env_theta"], fb_prev=fo, sanitize=0)
    assert beq(fb, fo)


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    sys.path.insert(0, os.path.dirname(HERE))
    import oracle  # noqa: E402
    from oracle import reference_shaders as R  # noqa: E402
    if not R.available():
        sys.exit("the reference's shaders are not built: `make -C oracle ref REFERENCE=<reference tree>`")
    out = {}
    make_pin(out, oracle, R)
    make_cuda(out, oracle, R)
    np.savez_compressed(PATH, **out)
    print("%s: %d outputs" % (PATH, len([k for k in out if k.endswith(":sha256")])))
