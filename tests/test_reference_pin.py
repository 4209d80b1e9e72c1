"""The oracle's external pin: the reference's OWN shader sources against the restatement.

camera.fs, bvh_test.fs, tracer.fs and draw.fs, compiled for the CPU behind the GLSL subset of oracle/glsl_cpu/
(`make -C oracle ref`, oracle/reference_shaders.py), were run on the inputs below and what they computed is stored in
tests/golden/reference_shaders/outputs.npz (generator: tests/golden/make_reference_outputs.py).  Every test puts
oracle/fspt_oracle.cpp (what all CUDA parity tests compare against) beside those outputs and demands identical bits:
control flow, operation order, constants, tie rules and the estimator of the restatement are thereby checked against
the reference's text, not against a reading of it.  What stays a model is what GLSL leaves to the platform (built-in
function precision, texture filtering arithmetic): oracle_math.h / oracle_texunit.h, shared by both sides.
"""
import os
import sys

import numpy as np
import pytest

from fspt_b200 import scenes
from oracle import reference_shaders as R

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_reference_outputs as golden  # noqa: E402


def beq(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.dtype.kind == "f":
        return bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))
    return bool(np.array_equal(a, b))


CAMERAS = [
    # W, H, eye, dir, fov_scale, (1 - 1/focal depth, aperture), randBase
    (64, 40, [0, 0.1, 2.5], [0, -0.05, -1], 0.5, [1 - 1 / 2.5, 0.02], 1234.5),
    (37, 53, [1.5, 2.0, -0.5], [-0.6, -0.7, 0.3], 0.8, [0.0, 0.0], 9999.75),      # odd size, pinhole
    (48, 48, [0, 3, 0], [0.0001, -1, 0.0], 0.3, [1 - 1 / 3.0, 0.25], 0.0),         # looking down: basisX near-degenerate
]
CAMERA_IDS = ["dof", "pinhole_odd", "down"]


@pytest.mark.parametrize("case", CAMERAS, ids=CAMERA_IDS)
def test_camera_fs(case, oracle_mod):
    W, H, P, I, fov, lens, rb = case
    name = CAMERA_IDS[CAMERAS.index(case)]
    po, do = oracle_mod.camera(W, H, P, I, fov, np.asarray(lens, np.float32), rb)
    golden.check("camera/%s/pos" % name, po)
    golden.check("camera/%s/dir" % name, do)


# config 5's resolution with the bunny camera
CAMERA_4K = (3840, 2160, scenes.BUNNY_CAMERA["eye"], scenes.BUNNY_CAMERA["dir"], scenes.BUNNY_CAMERA["fov_scale"],
             scenes.lens_features(scenes.BUNNY_CAMERA), 8191.25)


def test_camera_fs_at_3840x2160(oracle_mod):
    """config 5's resolution: camera.fs:38 seeds with randBase + gl_FragCoord.x * resolution.y + gl_FragCoord.y, above
    2^23 at the right edge, where f32 spacing is 1 and rows start to share seeds (and with them lens samples);
    restatement and shader must collide identically."""
    W, H, P, I, fov, lens, rb = CAMERA_4K
    po, do = oracle_mod.camera(W, H, P, I, fov, np.asarray(lens, np.float32), rb)
    golden.check("camera/3840x2160/pos", po)
    golden.check("camera/3840x2160/dir", do)
    # the collisions are real: 64 rows of the last column share lens samples, 64 rows of column 100 do not
    assert len(np.unique(po[:64, -1, 0])) < 64 and len(np.unique(po[:64, 100, 0])) == 64


def _primary(oracle_mod, sa, cam, W, H, rb):
    lens = np.asarray(scenes.lens_features(cam), np.float32)
    return oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rb)


def _random_rays(n, seed, scale=2.0):
    rng = np.random.default_rng(seed)
    pos = np.ones((n, 4), np.float32); d = np.ones((n, 4), np.float32)
    pos[:, :3] = rng.uniform(-scale, scale, (n, 3))
    v = rng.normal(size=(n, 3)); v /= np.linalg.norm(v, axis=1, keepdims=True)
    d[:, :3] = v
    # axis-parallel directions: zero components of either sign -> infinite slab inverses (tracer.fs:318)
    d[: n // 20, 0] = 0.0
    d[n // 20: n // 10, 1] = -0.0
    d[n // 10: n // 8, 2] = 0.0
    return pos, d


BVH_PRIMARY = (96, 64, 77.0)   # W, H, randBase of the primary rays of test_bvh_test_fs_index_t_count
BVH_RANDOM = (20000, 5)        # count, seed of its random rays


def _bvh_rays(oracle_mod, sa, cam):
    """(primary rays, random rays) of test_bvh_test_fs_index_t_count"""
    return _primary(oracle_mod, sa, cam, *BVH_PRIMARY), _random_rays(*BVH_RANDOM)


SCENES = {
    "bunny": lambda: scenes.bunny_class(subdiv=3, atlas_res=32, env_size=(128, 64)),
    "pbr_refractive": lambda: scenes.pbr_scene(atlas_res=16, subdiv=2, env_size=(64, 32)),
    "quad_kat": lambda: scenes.quad_scene(),
    "soup": lambda: scenes.sphere_soup(subdiv=3, n_soup=20000, seed=99, env_size=(64, 32)),
}


@pytest.mark.parametrize("name", list(SCENES))
def test_bvh_test_fs_index_t_count(name, oracle_mod):
    sa, cam = SCENES[name]()
    O = oracle_mod.Oracle(sa)
    for rays, (p4, d4) in zip(("primary", "random"), _bvh_rays(oracle_mod, sa, cam)):
        io, to, co, _ = O.bvh_test(p4, d4)
        key = "bvh_test/%s/%s/" % (name, rays)
        golden.check(key + "index", io)
        golden.check(key + "t", to)
        golden.check(key + "count", co)
        # the colour bvh_test.fs main() really writes (:230-231) is the count the restatement exports, times 0.001
        golden.check(key + "heat", co.astype(np.float32) * np.float32(0.001))
    assert (io >= 0).any() and (io < 0).any()


TRACER_CASES = [("bunny", 80, 48, 3), ("pbr_refractive", 64, 40, 3), ("quad_kat", 16, 16, 2), ("soup", 64, 36, 2)]
TRACER_SEED = 41  # of scenes.rand_bases


@pytest.mark.parametrize("name,W,H,ticks", TRACER_CASES)
def test_tracer_fs_accumulation(name, W, H, ticks, oracle_mod):
    """tracer.fs main() over consecutive ticks with the ping-ponged accumulation target (main.js:758-807)."""
    sa, cam = SCENES[name]()
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(ticks, TRACER_SEED)
    fo = None
    for k in range(ticks):
        pos, d = _primary(oracle_mod, sa, cam, W, H, rc[k])
        fo, st = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fo, sanitize=0, max_refractions=1 << 20)
        golden.check("tracer/%s/tick%d" % (name, k), fo)
    assert np.isfinite(fo).all() and fo[..., :3].max() > 0


THETAS = (0.0, 0.37, -1.25)
THETA_CASE = (48, 32, 3.5, 4242.0)  # W, H, camera randBase, tracer randBase of the bunny scene


def test_tracer_fs_rotated_environment(oracle_mod):
    sa, cam = SCENES["bunny"]()
    O = oracle_mod.Oracle(sa)
    W, H, rb_cam, rb_trace = THETA_CASE
    for theta in THETAS:
        pos, d = _primary(oracle_mod, sa, cam, W, H, rb_cam)
        fo, _ = O.trace(pos, d, W, H, 0, rb_trace, theta, sanitize=0)
        golden.check("tracer/bunny/theta%r" % theta, fo)


POSTS = [dict(exposure=1.0, saturation=1.0, denoise=False, max_sigma=2.0, scale=1.0),
         dict(exposure=1.7, saturation=0.6, denoise=True, max_sigma=2.0, scale=1.0),
         dict(exposure=0.4, saturation=1.4, denoise=True, max_sigma=0.5, scale=1.0),
         dict(exposure=1.0, saturation=1.0, denoise=True, max_sigma=2.0, scale=0.5)]
POST_IDS = ["post%d" % i for i in range(len(POSTS))]


def _draw_input(oracle_mod):
    sa, cam = SCENES["bunny"]()
    pos, d = _primary(oracle_mod, sa, cam, 64, 40, 12.0)
    fb, _ = oracle_mod.Oracle(sa).trace(pos, d, 64, 40, 0, 99.0, cam["env_theta"])
    fb[5, 7, :3] = 900.0  # a firefly for the 5x5 filter
    fb[20, 30, :3] = 0.0
    return fb


@pytest.mark.parametrize("post", POSTS)
def test_draw_fs(post, oracle_mod):
    golden.check("draw/%s" % POST_IDS[POSTS.index(post)], oracle_mod.draw(_draw_input(oracle_mod), **post))


@pytest.mark.skipif(not R.available(), reason="the blit shader of the reference's texture_packer.js is not in this "
                                              "repository; oracle/_ref/libfspt_ref.so is built only beside the reference tree")
@pytest.mark.parametrize("res,corrected,sw", [(64, True, None), (37, False, [2, 1, 0, 3]), (16, False, None),
                                              (128, True, [0, 0, 0, 3]), (53, True, [3, 2, 1, 0])])
def test_atlas_blit_shader_of_texture_packer_js(res, corrected, sw, oracle_mod):
    """The fragment shader inside texture_packer.js (:103-121, a JavaScript template string) with the GL state of
    :88-95,159-176 (REPEAT / CLAMP_TO_EDGE, LINEAR, SRGB8_ALPHA8 when `corrected`, swizzle uniform, RGBA8 read-back):
    restatement and the product's native blit against the shader text."""
    from fspt_b200 import capi
    rng = np.random.default_rng(2)
    img = rng.integers(0, 256, (37, 53, 4), dtype=np.uint8)  # odd, non-square, with alpha
    ref = R.pack_layer(img, res, corrected, sw)
    assert beq(oracle_mod.pack_layer(img, res, corrected, sw), ref)
    assert beq(capi.pack_layer(img, res, corrected, sw), ref)


def test_every_stored_output_is_also_checked_on_the_cuda_path():
    """tests/test_gpu_parity.py holds the CUDA path to every output stored for this pin, driving it from the case lists
    above.  A stored output those lists do not produce would be checked against the oracle only."""
    import test_gpu_parity as G
    with np.load(golden.PATH) as z:
        stored = {k.rsplit(":", 1)[0] for k in z.files}
    pinned = G.pinned_keys()
    assert len(pinned) == len(set(pinned))
    assert {k for k in stored if not k.startswith("cuda/")} == set(pinned)
