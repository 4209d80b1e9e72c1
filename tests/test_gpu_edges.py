"""The CUDA path at its limits, against the CPU oracle, bit for bit: the traversal stack filled to its last entry, the
refraction safety cap, crafted accumulators through the post pass (non-finite, negative, denormal and clamped values,
sum mode), degenerate rays, environment rotations far outside [0, 1) and the running mean across 2^24 ticks.

The tests marked `gpu` compare the two; the others check, without a GPU, that each oracle case really reaches the
limit it is about.
"""
import types

import numpy as np
import pytest

from fspt_b200 import capi, scenes

gpu = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bit_equal(got, ref, what):
    got, ref = np.ascontiguousarray(got), np.ascontiguousarray(ref)
    assert got.shape == ref.shape, "%s: shape %s, oracle %s" % (what, got.shape, ref.shape)
    if got.dtype.kind == "f":
        same = (bits(got) == bits(ref)) | (np.isnan(got) & np.isnan(ref))
    else:
        same = got == ref
    bad = int((~same).sum())
    if bad:
        i = np.argwhere(~same)[0]
        raise AssertionError("%s: %d of %d differ; first at %s: got %r oracle %r" %
                             (what, bad, same.size, tuple(i), got[tuple(i)], ref[tuple(i)]))


def _frame(ctx, cam, env_theta=None):
    return ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam),
                     cam["env_theta"] if env_theta is None else env_theta)


def _oracle_render(oracle_mod, O, cam, W, H, rc, rt, first_tick=0, fb=None, env_theta=None, **kw):
    """tracer.fs over len(rc) consecutive ticks from `first_tick` on: (accumulator, summed stats)"""
    tot = {}
    theta = cam["env_theta"] if env_theta is None else env_theta
    for k in range(len(rc)):
        pos, d = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        fb, st = O.trace(pos, d, W, H, first_tick + k, rt[k], theta, fb_prev=fb, **kw)
        for key, v in st.items():
            tot[key] = tot.get(key, 0) + v
    return fb, tot


@pytest.fixture(scope="module")
def tiny_bunny():
    return scenes.bunny_class(subdiv=2, atlas_res=16, env_size=(64, 32))


# ---------------------------------------------------------------------------------------------------------
# (a) the traversal stack at its limit
def chain_scene(levels, base):
    """A BVH of `levels` levels (the root counts as one): interior node k has a leaf as its left child and interior node
    k + 1 as its right one, the last interior node two leaves.  Every interior box is [-1, 1]^3; the leaf boxes,
    [-0.5, 0.5]^2 x [0.5, 1], lie behind it for a ray travelling along +z, so such a ray enters the interior child first
    and defers the leaf at every level: levels - 1 deferred children on top of the sentinel.  Each leaf holds 4 small
    triangles of its own (some rays hit one, others pass between them); the shading arrays are borrowed from `base`."""
    n = levels - 1
    rng = np.random.default_rng(levels)
    bvh = np.zeros((2 * n + 1, 9), np.float32)
    hdr = bvh.view(np.int32)
    tris = np.zeros((4 * levels, 9), np.float32)
    for i in range(n):
        hdr[2 * i, :3] = (2 * i + 1, 2 * i + 2, -1)
        bvh[2 * i, 3:9] = (-1, -1, -1, 1, 1, 1)
    for j, node in enumerate([2 * i + 1 for i in range(n)] + [2 * n]):
        hdr[node, 2] = 4 * j
        bvh[node, 3:9] = (-0.5, -0.5, 0.5, 0.5, 0.5, 1)
        for k in range(4):
            x, y = rng.uniform(-0.4, 0.4, 2)
            z = rng.uniform(0.55, 0.95)
            v = np.array([[x, y, z], [x + 0.2, y, z + 0.02], [x, y + 0.2, z - 0.02]], np.float32)
            v[:, :2] = np.clip(v[:, :2], -0.5, 0.5)
            tris[4 * j + k] = v.ravel()
    T = tris.shape[0]
    assert base.tris.shape[0] >= T
    return types.SimpleNamespace(bvh=bvh, tris=tris, mats=base.mats[:T], norms=base.norms[:T], uvs=base.uvs[:T],
                                 atlas=base.atlas, env=base.env, bins=base.bins, leaf_size=4)


AXIS_RAY = (np.array([[0.1, 0.2, -5.0, 1.0]], np.float32), np.array([[0.0, 0.0, 1.0, 1.0]], np.float32))
CHAIN_CAMERA = dict(eye=[0.0, 0.0, -5.0], dir=[0.0, 0.0, 1.0], fov_scale=0.2, env_theta=0.4, aperture=0.0, focal_depth=2.0)


def chain_rays(n=4000, seed=1):
    """Rays along +z, origins jittered over (and a little beyond) the boxes' cross-section, directions within ~1 degree"""
    rng = np.random.default_rng(seed)
    pos = np.ones((n, 4), np.float32)
    pos[:, :2] = rng.uniform(-1.1, 1.1, (n, 2))
    pos[:, 2] = -5.0
    v = np.c_[rng.normal(0.0, 0.02, (n, 2)), np.ones(n)]
    d = np.ones((n, 4), np.float32)
    d[:, :3] = v / np.linalg.norm(v, axis=1, keepdims=True)
    return np.r_[AXIS_RAY[0], pos], np.r_[AXIS_RAY[1], d]


def test_chain_at_the_stack_limit_fills_the_stack_in_the_oracle(tiny_bunny, oracle_mod):
    sa, _ = tiny_bunny
    O = oracle_mod.Oracle(chain_scene(64, sa))
    _, _, cnt, st = O.bvh_test(*AXIS_RAY)
    assert cnt[0] == 127 and st["stack_overflow"] == 0      # 63 interior nodes + 64 leaves, no push beyond 64 entries
    idx, _, cnt, st = O.bvh_test(*chain_rays())
    assert st["stack_overflow"] == 0 and (cnt == 127).sum() > 500
    assert (idx >= 0).any() and (idx[cnt == 127] < 0).any()  # hits and misses among the rays that fill the stack
    _, _, _, st = oracle_mod.Oracle(chain_scene(65, sa)).bvh_test(*AXIS_RAY)
    assert st["stack_overflow"] == 1                         # one level more than the reference's int stack[64] holds
    assert capi.debug_pack_scene(chain_scene(64, sa))["depth"] == 64


@gpu
@pytest.mark.parametrize("node_tex", [True, False], ids=["node_tex", "lsu"])
def test_traversal_stack_filled_to_its_last_entry(tiny_bunny, oracle_mod, monkeypatch, node_tex):
    """k_trace's 12 shared-memory entries plus its 52 local-memory spill entries, all in use; on both node-fetch paths.
    A tree one level deeper is refused by the upload (a host check) and the context stays usable."""
    if not node_tex:
        monkeypatch.setenv("FSPT_NO_NODE_TEX", "1")
    sa, _ = tiny_bunny
    deep = chain_scene(64, sa)
    O = oracle_mod.Oracle(deep)
    W, H = 64, 48
    ctx = capi.Context(W, H)
    try:
        with pytest.raises(capi.FsptError) as e:
            ctx.scene_upload(chain_scene(65, sa))
        assert e.value.code == -4 and "stack" in str(e.value)
        ctx.scene_upload(deep)
        pos, d = chain_rays()
        idx, t, cnt = ctx.debug_trace(pos, d)
        oi, ot, oc, st = O.bvh_test(pos, d)
        assert st["stack_overflow"] == 0 and oc[0] == 127
        assert_bit_equal(idx, oi, "hit index")
        assert_bit_equal(t, ot, "hit t")
        assert_bit_equal(cnt, oc, "visit count")
        cam = CHAIN_CAMERA
        rc, rt = scenes.rand_bases(2, 61)
        ctx.set_param(capi.PARAM_ANYHIT, 0)
        ctx.render(_frame(ctx, cam), 0, rc, rt)
        ofb, ost = _oracle_render(oracle_mod, O, cam, W, H, rc, rt)
        assert ost["stack_overflow"] == 0
        assert_bit_equal(ctx.read_accum()[..., :3], ofb[..., :3], "accumulator")
        s = ctx.stats()
        assert (s["last_rays"], s["last_node_visits"], s["last_leaf_visits"]) == \
            (ost["rays"], ost["node_visits"], ost["leaf_visits"])
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------
# (b) the refraction safety cap (tracer.fs:488 is unbounded in the reference)
CAP_SIZE = (96, 64)
CAPS = (0, 1, 2, 3, 64)


@pytest.fixture(scope="module")
def refractive():
    return scenes.pbr_scene(atlas_res=64, subdiv=2, env_size=(128, 64))


def test_refraction_cap_changes_the_oracle_image(refractive, oracle_mod):
    sa, cam = refractive
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(2, 7)
    ref, st = _oracle_render(oracle_mod, O, cam, *CAP_SIZE, rc, rt, max_refractions=64)
    assert st["capped"] == 0
    for cap in (0, 1):
        fb, st = _oracle_render(oracle_mod, O, cam, *CAP_SIZE, rc, rt, max_refractions=cap)
        assert st["capped"] > 0 and (bits(fb) != bits(ref)).any(-1).sum() > 100, cap


@gpu
def test_refraction_cap(refractive, oracle_mod):
    sa, cam = refractive
    W, H = CAP_SIZE
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(2, 7)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        for bad in (-1, 30001):
            with pytest.raises(capi.FsptError) as e:
                ctx.set_param(capi.PARAM_MAX_REFRACTIONS, bad)
            assert e.value.code == -1
        ctx.set_param(capi.PARAM_MAX_REFRACTIONS, 30000)
        fr = _frame(ctx, cam)
        for cap in CAPS:
            ctx.set_param(capi.PARAM_MAX_REFRACTIONS, cap)
            ctx.clear()
            before = ctx.stats()["capped_paths"]
            ctx.render(fr, 0, rc, rt)
            ofb, ost = _oracle_render(oracle_mod, O, cam, W, H, rc, rt, max_refractions=cap)
            assert_bit_equal(ctx.read_accum()[..., :3], ofb[..., :3], "accumulator, cap %d" % cap)
            s = ctx.stats()
            assert s["last_rays"] == ost["rays"], cap
            assert s["capped_paths"] - before == ost["capped"], cap
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------
# (c) crafted accumulators through k_post
POST_W, POST_H = 37, 23
SPECIAL = np.array([0.0, -0.0, 1e-40, -1e-40, 1.0, 1024.0, 3e38, np.inf, -np.inf, np.nan, -1.0, -3.5, 0.25, 7.0],
                   np.float32)


def crafted_accumulator(seed=3):
    rng = np.random.default_rng(seed)
    fb = rng.uniform(0.0, 2.0, (POST_H, POST_W, 4)).astype(np.float32)
    mask = rng.random((POST_H, POST_W, 4)) < 0.3
    fb[mask] = rng.choice(SPECIAL, int(mask.sum()))
    fb[8:13, 8:13, :3] = 50.0                     # a zero-luma centre in a bright 5x5 block (draw.fs divides by it)
    fb[10, 10, :3] = 0.0
    fb[14:17, 29:32, :3] = 9.0
    fb[15, 30, :3] = (-0.7152, 0.2126, 0.0)      # luma 0 from non-zero colours
    fb[1:7, 18:27, :3] = 0.1                      # flat blocks: the variance can round below zero
    fb[16:22, 2:9, :3] = 0.3
    fb[16:22, 12:18, :3] = 1024.0
    for y, x in ((0, 0), (0, POST_W - 1), (POST_H - 1, 0), (POST_H - 1, POST_W - 1), (0, 17), (11, 0), (POST_H - 1, 20),
                 (6, POST_W - 1)):
        fb[y, x, :3] = 500.0                      # bright pixels on the borders and corners
    return fb


POST_GRID = [dict(exposure=e, saturation=s, denoise=dn, max_sigma=ms, scale=sc)
             for e in (1.0, 0.0, 3.5) for s in (1.0, 0.0, 2.0) for sc in (1.0, 0.5, 0.3, 1.5, 2.0)
             for dn, ms in ((False, 2.0), (True, 2.0), (True, 0.5), (True, 0.0))]


@gpu
def test_post_pass_on_crafted_accumulators(oracle_mod):
    fb = crafted_accumulator()
    ctx = capi.Context(POST_W, POST_H)
    try:
        ctx.write_accum(fb, 1)
        assert_bit_equal(ctx.read_accum(), fb, "accumulator round trip")
        for kw in POST_GRID:
            assert_bit_equal(ctx.resolve(**kw), oracle_mod.draw(fb, **kw), "rgba8 %r" % (kw,))
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------
# (d) sum-mode resolve on one GPU: every pixel divided by its own sample count, 0 samples -> black
def _mean_of_sums(fb):
    with np.errstate(all="ignore"):
        q = fb[..., :3] / fb[..., 3:4]
    out = np.zeros_like(fb)
    out[..., :3] = np.where(fb[..., 3:4] > 0, q, np.float32(0.0))
    return out


SUM_POSTS = [dict(denoise=dn, scale=sc, exposure=1.3) for dn in (False, True) for sc in (1.0, 0.5)]


@gpu
def test_sum_mode_resolve_with_uncovered_pixels(small_bunny, oracle_mod):
    sa, cam = small_bunny
    W, H = 64, 48
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(3, 17)
    tiles = [((0, 0, 40, 20), 2), ((24, 20, 40, 17), 3)]  # rows 37..47 and the rest of the frame: no sample at all
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        ctx.set_accum_mode(1)
        ctx.clear()
        fr = _frame(ctx, cam)
        for rect, n in tiles:
            ctx.set_tile(*rect)
            ctx.render(fr, 0, rc[:n], rt[:n])
        cols = []
        for k in range(3):
            pos, d = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
            cols.append(O.trace(pos, d, W, H, 0, rt[k], cam["env_theta"], want_color=True)[1])
        ref = np.zeros((H, W, 4), np.float32)
        for (x0, y0, w, h), n in tiles:
            for k in range(n):
                ref[y0:y0 + h, x0:x0 + w, :3] += cols[k][y0:y0 + h, x0:x0 + w, :3]
            ref[y0:y0 + h, x0:x0 + w, 3] = n
        assert (ref[..., 3] == 0).any()
        assert_bit_equal(ctx.read_accum(), ref, "sum accumulator")
        mean = _mean_of_sums(ref)
        for kw in SUM_POSTS:
            assert_bit_equal(ctx.resolve(**kw), oracle_mod.draw(mean, **kw), "rgba8 %r" % (kw,))
        # crafted sums: sample counts 0, 1, 3 and 2^24 under every kind of value
        fb = np.ascontiguousarray(np.tile(crafted_accumulator(5), (3, 2, 1))[:H, :W])
        fb[..., 3] = np.resize(np.array([0.0, 1.0, 3.0, 2.0 ** 24], np.float32), (H, W))
        ctx.write_accum(fb, 0)
        mean = _mean_of_sums(fb)
        for kw in SUM_POSTS:
            assert_bit_equal(ctx.resolve(**kw), oracle_mod.draw(mean, **kw), "crafted sums, rgba8 %r" % (kw,))
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------
# (e) degenerate rays
def degenerate_rays(sa, seed=9):
    rng = np.random.default_rng(seed)
    P, D = [], []

    def add(p, d):
        p = np.asarray(p, np.float32).reshape(-1, 3)
        d = np.asarray(d, np.float32).reshape(-1, 3)
        p, d = np.broadcast_arrays(p, d)
        P.append(p)
        D.append(d)

    n = 512
    v = rng.normal(size=(n, 3))
    base_p = rng.uniform(-1.5, 1.5, (n, 3)).astype(np.float32)
    base_d = (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)
    add(base_p, base_d)
    for bad in (np.nan, np.inf, -np.inf):         # a non-finite component in the origin or the direction
        for c in range(3):
            p, d = base_p.copy(), base_d.copy()
            p[:, c] = bad
            add(p, base_d)
            d[:, c] = bad
            add(base_p, d)
    add(base_p, [0.0, 0.0, 0.0])                  # zero directions
    add(base_p, [-0.0, 0.0, -0.0])
    for dd in ([1e-40, 0.0, 0.0], [0.0, -1e-45, 0.0], [1e-40, -3e-39, 1e-42], [1e-40, 1.0, 0.0], [0.7, 1e-40, -0.7],
               [-1e-38, 1e-39, 1.0]):            # denormal components
        add(base_p, dd)
    # origins on faces of node boxes, with generic and axis-parallel directions ((b - o) * (1 / 0) = 0 * inf = NaN)
    boxes = np.ascontiguousarray(sa.bvh, np.float32).reshape(-1, 9)[:, 3:9]
    pick = boxes[rng.integers(0, boxes.shape[0], 64)]
    for face in range(6):
        lo, hi = pick[:, :3], pick[:, 3:]
        p = lo + (hi - lo) * rng.random((64, 3)).astype(np.float32)
        p[:, face % 3] = pick[:, face]
        add(p, base_d[:64])
        axis = np.zeros((64, 3), np.float32)
        axis[:, face % 3] = 1.0 if face < 3 else -1.0
        add(p, axis)
        axis[:, face % 3] = 0.0
        axis[:, (face + 1) % 3] = -1.0
        add(p, axis)
    # rays through vertices and edges of triangles (u = 0, v = 0, u + v = 1), straight down and slanted
    tris = np.ascontiguousarray(sa.tris, np.float32).reshape(-1, 3, 3)
    sel = tris[rng.integers(0, tris.shape[0], 48)]
    pts = [sel[:, 0], sel[:, 1], sel[:, 2], (sel[:, 0] + sel[:, 1]) * 0.5, (sel[:, 1] + sel[:, 2]) * 0.5,
           (sel[:, 0] + sel[:, 2]) * 0.5, sel[:, 1] * 0.25 + sel[:, 2] * 0.75]
    for q in pts:
        q = q.astype(np.float32)
        add(q + np.float32([0.0, 1.0, 0.0]), [0.0, -1.0, 0.0])
        add(q + np.float32([0.0, -1.0, 0.0]), [0.0, 1.0, 0.0])
        add(q + np.float32([0.5, 1.0, -0.25]), np.float32([-0.5, -1.0, 0.25]))
    # rays parallel to a triangle's plane: along its edges, from inside the plane and beside it
    e1 = (sel[:, 1] - sel[:, 0]).astype(np.float32)
    e2 = (sel[:, 2] - sel[:, 0]).astype(np.float32)
    for e in (e1, e2, e2 - e1):
        add(sel[:, 0] - e, e)
        add(sel[:, 0] - e + np.float32([0.0, 1e-3, 0.0]), e)
    add([[x, 0.0, z] for x in (-0.75, -0.5, 0.0, 0.5) for z in (-0.5, 0.0, 0.25)], [1.0, 0.0, 0.0])   # in y = 0
    add([[x, 0.0, z] for x in (-0.75, -0.5, 0.0, 0.5) for z in (-0.5, 0.0, 0.25)], [0.0, 0.0, -1.0])
    # the axis-aligned quad of quad_scene (y = 0, [-0.5, 0.5]^2): its corners, edges and shared diagonal, exactly
    g = np.float32([-0.5, -0.25, 0.0, 0.25, 0.5])
    grid = np.array([[x, 1.0, z] for x in g for z in g], np.float32)
    add(grid, [0.0, -1.0, 0.0])
    add(grid * np.float32([1.0, -1.0, 1.0]), [0.0, 1.0, 0.0])
    pos = np.ones((sum(len(p) for p in P), 4), np.float32)
    d = np.ones_like(pos)
    pos[:, :3] = np.concatenate(P)
    d[:, :3] = np.concatenate(D)
    return pos, d


@gpu
@pytest.mark.parametrize("scene", ["small_bunny", "quad"])
def test_degenerate_rays(scene, small_bunny, oracle_mod):
    sa, _ = small_bunny if scene == "small_bunny" else scenes.quad_scene()
    pos, d = degenerate_rays(sa)
    ctx = capi.Context(16, 16)
    try:
        ctx.scene_upload(sa)
        idx, t, cnt = ctx.debug_trace(pos, d)
    finally:
        ctx.close()
    oi, ot, oc, _ = oracle_mod.Oracle(sa).bvh_test(pos, d)
    assert (oi >= 0).any()
    assert_bit_equal(idx, oi, "hit index")
    assert_bit_equal(t, ot, "hit t")
    assert_bit_equal(cnt, oc, "visit count")


# ---------------------------------------------------------------------------------------------------------
# (f) environment rotations and the running mean across 2^24 ticks
ENV_SCENES = {
    "env96x48": lambda: scenes.bunny_class(subdiv=3, atlas_res=24, env_size=(96, 48)),   # wrap by modulo, not by a mask
    "env128x64": lambda: scenes.bunny_class(subdiv=3, atlas_res=32, env_size=(128, 64)),
}
# -2e7 puts the texel coordinate beyond the +-1e9 guard of coord_to_i32
THETAS = (-1.25, 123.456, -2e7)


@gpu
@pytest.mark.parametrize("env", list(ENV_SCENES))
def test_environment_rotation_extremes(env, oracle_mod):
    sa, cam = ENV_SCENES[env]()
    W, H = 64, 40
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(2, 71)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        for theta in THETAS:
            ctx.clear()
            ctx.render(_frame(ctx, cam, theta), 0, rc, rt)
            ofb, _ = _oracle_render(oracle_mod, O, cam, W, H, rc, rt, env_theta=theta)
            assert_bit_equal(ctx.read_accum()[..., :3], ofb[..., :3], "accumulator, env_theta %r" % theta)
    finally:
        ctx.close()


@gpu
def test_running_mean_across_two_to_the_24_ticks(oracle_mod):
    """(color + prev * tick) / (tick + 1) with float(tick) no longer exact above 2^24 (tracer.fs:517)."""
    sa, cam = ENV_SCENES["env128x64"]()
    W, H = 48, 32
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(6, 73)
    start = 2 ** 24 - 2
    prev, _ = _oracle_render(oracle_mod, O, cam, W, H, rc[:2], rt[:2])
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        ctx.write_accum(prev, start)
        ctx.render(_frame(ctx, cam), start, rc[2:], rt[2:])
        ofb, _ = _oracle_render(oracle_mod, O, cam, W, H, rc[2:], rt[2:], first_tick=start, fb=prev)
        assert_bit_equal(ctx.read_accum()[..., :3], ofb[..., :3], "accumulator")
    finally:
        ctx.close()
