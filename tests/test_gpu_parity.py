"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on identical inputs.

Bars (BASELINE.md section 4 / north star):
  * primary-hit records (index, t, count) of the bvh_test.fs traversal: BIT-EXACT;
  * camera rays, per-sample radiance, running-mean accumulator and RGBA8 post-pass: the CUDA kernels
    implement the same FSPT-DM2 arithmetic as the oracle, so these are asserted bit-exact as well
    (stated tolerance: 0 ulp; a mismatch-rate report is printed if that ever fails).
"""
import os
import sys

import numpy as np
import pytest

from fspt_b200 import capi, scenes

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_reference_outputs as golden  # noqa: E402

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bit_equal(got, ref, what):
    got, ref = np.ascontiguousarray(got), np.ascontiguousarray(ref)
    if got.dtype.kind == "f":
        same = (bits(got) == bits(ref)) | (np.isnan(got) & np.isnan(ref))
    else:
        same = got == ref
    bad = int((~same).sum())
    if bad:
        i = np.argwhere(~same)[0]
        raise AssertionError("%s: %d of %d differ; first at %s: got %r ref %r" %
                             (what, bad, same.size, tuple(i), got[tuple(i)], ref[tuple(i)]))


@pytest.fixture(scope="module")
def ctx_small(small_bunny):
    sa, cam = small_bunny
    ctx = capi.Context(160, 96)
    ctx.scene_upload(sa)
    yield ctx
    ctx.close()


def _frame(ctx, cam):
    return ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])


def test_dm_math_matches_oracle(ctx_small, oracle_mod):
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.uniform(-1e7, 1e7, 100000), rng.uniform(-8, 8, 100000), [0.0, -0.0, 1e-30, 3.4e38]]).astype(np.float32)
    for fn in ("sin", "cos"):
        assert_bit_equal(ctx_small.debug_math(fn, x), oracle_mod.dm_eval(fn, x), fn)
    assert_bit_equal(ctx_small.debug_math("sincos_s", x), oracle_mod.dm_eval("sin", x), "sincos.s")
    assert_bit_equal(ctx_small.debug_math("sincos_c", x), oracle_mod.dm_eval("cos", x), "sincos.c")
    a = rng.uniform(-1.01, 1.01, 100000).astype(np.float32)
    b = rng.uniform(-1, 1, 100000).astype(np.float32)
    assert_bit_equal(ctx_small.debug_math("atan2", a, b), oracle_mod.dm_eval("atan2", a, b), "atan2")
    assert_bit_equal(ctx_small.debug_math("asin", a), oracle_mod.dm_eval("asin", a), "asin")
    e = rng.uniform(-150, 130, 100000).astype(np.float32)
    assert_bit_equal(ctx_small.debug_math("exp2", e), oracle_mod.dm_eval("exp2", e), "exp2")
    p = rng.uniform(0, 2, 100000).astype(np.float32)
    q = rng.uniform(0.1, 3, 100000).astype(np.float32)
    assert_bit_equal(ctx_small.debug_math("pow", p, q), oracle_mod.dm_eval("pow", p, q), "pow")


def test_camera_and_primary_hits_bit_exact(ctx_small, small_bunny, oracle_mod):
    sa, cam = small_bunny
    O = oracle_mod.Oracle(sa)
    for rb in (1234.5, 9876.25):
        idx, t, cnt, pos, d = ctx_small.debug_primary(_frame(ctx_small, cam), rb)
        opos, odir = oracle_mod.camera(160, 96, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rb)
        assert_bit_equal(pos, opos, "camera pos")
        assert_bit_equal(d, odir, "camera dir")
        oi, ot, oc, st = O.bvh_test(opos, odir)
        assert_bit_equal(idx, oi, "hit index")
        assert_bit_equal(t, ot, "hit t")
        assert_bit_equal(cnt, oc, "visit count")
        assert (oi >= 0).mean() > 0.3


def test_debug_trace_random_rays(ctx_small, small_bunny, oracle_mod):
    sa, _ = small_bunny
    O = oracle_mod.Oracle(sa)
    rng = np.random.default_rng(11)
    n = 50000
    pos = np.ones((n, 4), np.float32)
    pos[:, :3] = rng.uniform(-1.5, 1.5, (n, 3))
    d = np.ones((n, 4), np.float32)
    v = rng.normal(size=(n, 3))
    d[:, :3] = (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)
    d[:100, 0] = 0.0   # axis-parallel components: 1/0 = inf slabs
    d[100:200, 1] = -0.0
    idx, t, cnt = ctx_small.debug_trace(pos, d)
    oi, ot, oc, st = O.bvh_test(pos, d)
    assert_bit_equal(idx, oi, "hit index")
    assert_bit_equal(t, ot, "hit t")
    assert_bit_equal(cnt, oc, "visit count")
    s = ctx_small.stats()
    assert s["rays"] >= n


def test_radiance_accumulator_bit_exact(ctx_small, small_bunny, oracle_mod):
    sa, cam = small_bunny
    O = oracle_mod.Oracle(sa)
    W, H, N = 160, 96, 6
    rc, rt = scenes.rand_bases(N, 42)
    ctx_small.clear()
    ctx_small.render(_frame(ctx_small, cam), 0, rc, rt)
    fb = ctx_small.read_accum()
    last = ctx_small.debug_last_color()
    ofb = None
    rays = 0
    for k in range(N):
        pos, d = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        ofb, ocol, st = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=ofb, want_color=True)
        rays += st["rays"]
    assert_bit_equal(last[..., :3], ocol[..., :3], "last sample colour")
    assert_bit_equal(fb[..., :3], ofb[..., :3], "accumulator")
    s = ctx_small.stats()
    assert s["last_rays"] == rays
    # split renders continue the same running mean
    ctx_small.clear()
    ctx_small.render(_frame(ctx_small, cam), 0, rc[:2], rt[:2])
    ctx_small.render(_frame(ctx_small, cam), 2, rc[2:], rt[2:])
    assert_bit_equal(ctx_small.read_accum()[..., :3], ofb[..., :3], "accumulator (split)")


def test_post_pass_bit_exact(ctx_small, small_bunny, oracle_mod):
    sa, cam = small_bunny
    rc, rt = scenes.rand_bases(3, 5)
    ctx_small.clear()
    ctx_small.render(_frame(ctx_small, cam), 0, rc, rt)
    fb = ctx_small.read_accum()
    for kw in (dict(), dict(denoise=True, max_sigma=2.0), dict(exposure=1.7, saturation=0.6), dict(denoise=True, exposure=0.5, saturation=1.3)):
        got = ctx_small.resolve(**kw)
        ref = oracle_mod.draw(fb, **kw)
        assert_bit_equal(got, ref, "rgba8 %r" % (kw,))


# ---------------------------------------------------------------------------------------------------------
# BASELINE.json full sizes: whole frames against the oracle, bit for bit
def _full_frame_check(oracle_mod, sa, cam, W, H, n, seed):
    O = oracle_mod.Oracle(sa)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        rc, rt = scenes.rand_bases(n, seed)
        idx, t, cnt, pos, d = ctx.debug_primary(fr, rc[0])
        opos, odir = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[0])
        assert_bit_equal(pos, opos, "camera pos")
        assert_bit_equal(d, odir, "camera dir")
        oi, ot, oc, st = O.bvh_test(opos, odir)
        assert_bit_equal(idx, oi, "hit index")
        assert_bit_equal(t, ot, "hit t")
        assert_bit_equal(cnt, oc, "visit count")
        ctx.set_param(capi.PARAM_ANYHIT, 0)  # full closest-hit traversal for every ray, like the reference
        ctx.clear()
        ctx.render(fr, 0, rc, rt)
        fb = ctx.read_accum()
        ofb, rays, nodes, leaves = None, 0, 0, 0
        for k in range(n):
            p, dd = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
            ofb, s2 = O.trace(p, dd, W, H, k, rt[k], cam["env_theta"], fb_prev=ofb)
            rays += s2["rays"]; nodes += s2["node_visits"]; leaves += s2["leaf_visits"]
        assert_bit_equal(fb[..., :3], ofb[..., :3], "accumulator")
        s = ctx.stats()
        # the device-side V / L counters that feed bench.py's algorithmic bytes equal the oracle's
        assert (s["last_rays"], s["last_node_visits"], s["last_leaf_visits"]) == (rays, nodes, leaves)
        assert_bit_equal(ctx.resolve(denoise=True), oracle_mod.draw(ofb, denoise=True), "rgba8")
        # default mode: hit-or-miss rays stop at their first intersection -- same image, same ray count, fewer visits
        ctx.set_param(capi.PARAM_ANYHIT, 1)
        ctx.clear()
        ctx.render(fr, 0, rc, rt)
        assert_bit_equal(ctx.read_accum()[..., :3], ofb[..., :3], "accumulator (any-hit)")
        s = ctx.stats()
        assert s["last_rays"] == rays and s["last_node_visits"] <= nodes and s["last_leaf_visits"] <= leaves
    finally:
        ctx.close()


def test_full_size_bunny_frame_bit_exact(oracle_mod):
    """BASELINE configs[1] exactly as bench.py renders it: 1280x720, 81,920-triangle bunny-class mesh + the two textured
    quads, 2048x2048 atlas (11 layers), 2048x1024 environment."""
    sa, cam = scenes.bunny_class(subdiv=6, atlas_res=2048)
    assert sa.atlas.shape[1] == 2048
    _full_frame_check(oracle_mod, sa, cam, 1280, 720, 2, 3)


def test_million_triangle_soup_bit_exact(oracle_mod):
    """BASELINE configs[2]: 1 M triangles (icosphere + soup), 1280x720, primary + 4 bounces."""
    sa, cam = scenes.sphere_soup()
    assert sa.n_tris == 1000000
    _full_frame_check(oracle_mod, sa, cam, 1280, 720, 1, 5)


def test_refractive_pbr_scene_bit_exact(oracle_mod):
    """BASELINE configs[3] features: four texture maps per prop + a refractive prop (dielectric >= 0, free bounces)."""
    sa, cam = scenes.pbr_scene(atlas_res=256, subdiv=4)
    _full_frame_check(oracle_mod, sa, cam, 480, 270, 3, 9)
    assert (sa.mats[:, 10] >= 0).any()


def test_refractive_pbr_scene_full_size_bit_exact(oracle_mod):
    """BASELINE configs[3] at its own size: 1920x1080, atlasRes 2048, refraction (paths beyond NUM_BOUNCES go through the
    pipelined live-path poll of render_wave)."""
    sa, cam = scenes.pbr_scene(atlas_res=2048)
    assert sa.atlas.shape[1] == 2048 and (sa.mats[:, 10] >= 0).any()
    _full_frame_check(oracle_mod, sa, cam, 1920, 1080, 2, 13)


def test_ten_million_triangles_at_4k_bit_exact(oracle_mod):
    """BASELINE configs[4] geometry and resolution: 10 M triangles (subdiv-8 icosphere + 8.69 M soup, seed 4321) at
    3840x2160, 1 sample: camera rays (gl_FragCoord seeds beyond 2^22, where `seed += 0.2113` stalls in f32,
    camera.fs:19,38), primary (index, t, count), the accumulator with and without any-hit, and the device V / L counters
    against the CPU oracle.  The BVH (0.7 GB of nodes + triangles) no longer fits the L2."""
    sa, cam = scenes.sphere_soup(subdiv=8, n_soup=10000000 - 1310720, seed=4321)
    assert sa.n_tris == 10000000 and sa.depth <= 64
    _full_frame_check(oracle_mod, sa, cam, 3840, 2160, 1, 17)


def test_node_records_through_the_lsu_path_bit_exact(oracle_mod, monkeypatch, small_bunny):
    """k_trace<.., NODE_TEX = false>: the instantiation used when the node array exceeds the 2^27-texel limit of a linear
    texture (> 33 M interior nodes) -- forced here on a small scene."""
    monkeypatch.setenv("FSPT_NO_NODE_TEX", "1")
    sa, cam = small_bunny
    _full_frame_check(oracle_mod, sa, cam, 160, 96, 2, 19)


REF_W, REF_H, REF_N = 128, 72, 4
REF_POST = dict(exposure=1.2, saturation=0.9, denoise=True, max_sigma=2.0)


def test_cuda_against_the_reference_shaders_themselves(small_bunny):
    """No restatement in between: the CUDA path against what the reference's own camera.fs, bvh_test.fs, tracer.fs and
    draw.fs, compiled for the CPU, computed on the same inputs (tests/golden/reference_shaders/outputs.npz, generator
    tests/golden/make_reference_outputs.py).  Camera rays, primary hits (index, t, count), the running-mean accumulator
    over 4 ticks and the RGBA8 post-pass."""
    sa, cam = small_bunny
    W, H, N = REF_W, REF_H, REF_N
    rc, rt = scenes.rand_bases(N, 29)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        idx, t, cnt, pos, d = ctx.debug_primary(fr, float(rc[0]))
        golden.check("cuda/camera/pos", pos)
        golden.check("cuda/camera/dir", d)
        golden.check("cuda/bvh_test/index", idx)
        golden.check("cuda/bvh_test/t", t)
        golden.check("cuda/bvh_test/count", cnt)
        ctx.clear()
        ctx.set_param(capi.PARAM_SANITIZE_NAN, 0)  # the reference lets NaN stick (tracer.fs:515-517)
        ctx.render(fr, 0, rc, rt)
        golden.check("cuda/tracer/accum_rgb", ctx.read_accum()[..., :3])
        golden.check("cuda/draw/rgba8", ctx.resolve(**REF_POST))
    finally:
        ctx.close()


def test_non_power_of_two_atlas_and_environment_bit_exact(oracle_mod):
    """Texture sizes that are not powers of two: the REPEAT wrap takes the modulo path instead of a mask and sampleEnv's
    divisions by the environment size stay divisions (for powers of two they are multiplications by the exact
    reciprocal) -- a 24-texel atlas and a 96x48 environment against the oracle."""
    sa, cam = scenes.bunny_class(subdiv=3, atlas_res=24, env_size=(96, 48))
    assert sa.atlas.shape[1] == 24 and sa.env.shape[:2] == (48, 96)
    _full_frame_check(oracle_mod, sa, cam, 160, 96, 3, 23)
