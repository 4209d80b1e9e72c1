"""A long-lived context against fresh ones: scene swaps, context settings and adaptive checkpoints, bit for bit.

A context keeps its device buffers, arrays, texture objects, tables and constants across uploads and reuses what fits
(fit_scene / publish_scene / fit_atlas / publish_atlas in fspt_api.cu).  PathTracer, the N-API shim and bench.py's
end-to-end loop all render many scenes through one context, so anything stale after a swap would show up there only.

  * walk_scenes() is one fixed list of small scenes in which every dimension the kept storage depends on changes, up and down:
    triangles, interior nodes and depth past the kept capacity and below it, a root that is a leaf, the environment's
    width, height and power-of-two-ness (and a 1-bin environment), the radiance bin count, the atlas resolution, layer
    count and textured-material count, and a dielectric.  Each walk renders every scene in order through one context
    and compares, per scene, with a fresh context and with the CPU oracle: accumulator (running mean and sum mode), last
    sample colour, primary hits and camera rays, per-render counters and the post pass.  The walks differ in how the
    scene arrives (synchronous, asynchronous, page-locked) and in the upload knobs switched between scenes; each walk
    also meets one refused upload.
  * Settings of the context (any-hit, refraction cap, tile, sum mode) apply to the scene after a swap.
  * Adaptive sampling's state moves between contexts: accumulator + moment + next tick continue to the same bits, and
    fspt_clear starts the moment from zero.

The CPU test at the end checks from the scene arrays alone that the walk covers every dimension it claims to.
"""
import copy
import functools

import numpy as np
import pytest

from fspt_b200 import capi, scenes, procedural as pr

import test_gpu_adaptive as adaptive  # the shared builders and helpers of the other GPU tests
import test_gpu_edges as edges
import test_gpu_shading_matrix as matrix

gpu = pytest.mark.gpu
W, H, TICKS = 64, 48, 2
E_STATE, E_LIMIT = -3, -4
POSTS = (dict(denoise=True), dict(exposure=1.3, saturation=0.7, denoise=True, scale=0.5))  # by accumulation mode
assert_bit_equal = edges.assert_bit_equal


# ---------------------------------------------------------------------------------------------------------------------
# the walk
def _soup_with_one_bin():
    """An untextured soup under a 1 x 1 constant environment: one radiance bin."""
    sa, cam = scenes.sphere_soup(subdiv=2, n_soup=1500, env_size=(32, 16))
    sa = copy.copy(sa)
    sa.env = pr.constant_environment(1, 1, 0.8)
    sa.bins = capi.env_bins(sa.env)
    return sa, cam


@functools.lru_cache(maxsize=None)
def walk_scenes():
    """[(name, scene arrays, camera)].  The first scene has no dielectric, so a render that kept the first upload's
    refraction handling would cut the refractive paths of later scenes short."""
    bunny2 = scenes.bunny_class(subdiv=2, atlas_res=16, env_size=(96, 48))
    bunny3 = scenes.bunny_class(subdiv=3, atlas_res=32, env_size=(128, 64))
    quad = scenes.quad_scene(env_size=(64, 32))
    chain_cam = dict(edges.CHAIN_CAMERA)
    uvs, uvs_cam, _ = matrix.build_case("uvs", 32)
    diel, diel_cam, _ = matrix.build_case("dielectrics", 24)
    return [
        ("bunny_s2_r16", *bunny2),
        ("chain64_r16", edges.chain_scene(64, bunny2[0]), chain_cam),   # same atlas: the interleaved array is kept
        ("quad", *quad),                                                # root is a leaf, everything shrinks
        ("pbr_r32", *scenes.pbr_scene(atlas_res=32, subdiv=1, env_size=(128, 64))),
        ("bunny_s3_r32", *bunny3),                                      # same resolution, other textured materials
        ("uvs_r32", uvs, uvs_cam),                                      # same resolution and layer count, other tables
        ("pbr_r16", *scenes.pbr_scene(atlas_res=16, subdiv=2, env_size=(64, 48))),  # same env width, taller, not pow2
        ("quad_again", *quad),                                          # same env width, shorter, pow2 again
        ("chain64_r32", edges.chain_scene(64, bunny3[0]), chain_cam),   # a leaf root, then 64 levels
        ("soup_env1", *_soup_with_one_bin()),
        ("dielectrics_r24", diel, diel_cam),
        ("bunny_s1_r32", *scenes.bunny_class(subdiv=1, atlas_res=32, env_size=(128, 64))),
        ("bunny_s3_r32_again", *bunny3),                                # same atlas shape and materials, more geometry
    ]


REFUSED_BEFORE = 7  # the walk's refused upload comes right before this step


def _step(name):
    return next(i for i, step in enumerate(walk_scenes()) if step[0] == name)


def _refused():
    return edges.chain_scene(65, walk_scenes()[0][1])  # one level more than the traversal stack holds


# upload knobs, switched between consecutive scenes of the "knobs" walk (read by each upload)
KNOBS = ({}, {"FSPT_PLAIN_ATLAS": "1"}, {"FSPT_ATLAS_INTERLEAVE": "gpu"},
         {"FSPT_NO_NODE_TEX": "1", "FSPT_ATLAS_INTERLEAVE": "cpu"}, {"FSPT_PLAIN_ATLAS": "1", "FSPT_NO_NODE_TEX": "1"})
KNOB_NAMES = ("FSPT_PLAIN_ATLAS", "FSPT_ATLAS_INTERLEAVE", "FSPT_NO_NODE_TEX")
# how the scenes of a walk arrive: upload_wait per step (cycled), page-locked atlas and environment, knobs
WALKS = {
    "sync": dict(waits=(True,)),
    "async": dict(waits=(False,)),
    "pinned": dict(waits=(True, False), pinned=True),
    "knobs": dict(waits=(True, False, False), knobs=True),
}


def _frame(ctx, cam):
    return ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])


def _rand(i):
    return scenes.rand_bases(TICKS, 100 + i)


# ---------------------------------------------------------------------------------------------------------------------
# the two references of a step: the oracle, and a fresh context that has only that scene
@functools.lru_cache(maxsize=None)
def oracle_step(i):
    import oracle
    _, sa, cam = walk_scenes()[i]
    O = oracle.Oracle(sa)
    rc, rt = _rand(i)
    fb, total, cols = None, dict(rays=0, node_visits=0, leaf_visits=0, capped=0), []
    for k in range(TICKS):
        pos, d = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        fb, col, st = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fb, want_color=True)
        cols.append(col)
        for key in total:
            total[key] += st[key]
    sums = np.zeros((H, W, 4), np.float32)
    for col in cols:
        sums[..., :3] += col[..., :3]
    sums[..., 3] = TICKS
    pos, d = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[0])
    idx, t, cnt, _ = O.bvh_test(pos, d)
    return dict(accum=(fb, sums), last=cols[-1], counters=total, primary=(idx, t, cnt, pos, d),
                rgba8=(oracle.draw(fb, **POSTS[0]), oracle.draw(edges._mean_of_sums(sums), **POSTS[1])))


def _render_step(ctx, i, mode):
    """Render step i in accumulation mode `mode` on a context that holds scene i: everything the walk compares."""
    _, _, cam = walk_scenes()[i]
    rc, rt = _rand(i)
    fr = _frame(ctx, cam)
    ctx.set_accum_mode(mode)
    ctx.clear()
    capped0 = ctx.stats()["capped_paths"]
    ctx.render(fr, 0, rc, rt)
    out = dict(accum=ctx.read_accum(), last=ctx.debug_last_color())
    s = ctx.stats()
    out["counters"] = dict(rays=s["last_rays"], node_visits=s["last_node_visits"], leaf_visits=s["last_leaf_visits"],
                           capped=s["capped_paths"] - capped0)
    out["rgba8"] = ctx.resolve(**POSTS[mode])
    out["primary"] = ctx.debug_primary(fr, rc[0])
    return out


@functools.lru_cache(maxsize=None)
def fresh_step(i, mode):
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(walk_scenes()[i][1])
        ctx.set_param(capi.PARAM_ANYHIT, 0)
        return _render_step(ctx, i, mode)
    finally:
        ctx.close()


def _check_step(got, i, mode, what):
    ref, orc = fresh_step(i, mode), oracle_step(i)
    for key in ("accum", "last", "rgba8"):
        assert_bit_equal(got[key], ref[key], "%s: %s against a fresh context" % (what, key))
    for g, r, name in zip(got["primary"], ref["primary"], ("index", "t", "count", "pos", "dir")):
        assert_bit_equal(g, r, "%s: primary %s against a fresh context" % (what, name))
    assert got["counters"] == ref["counters"], (what, got["counters"], ref["counters"])
    acc = got["accum"] if mode else got["accum"][..., :3]
    assert_bit_equal(acc, orc["accum"][mode] if mode else orc["accum"][0][..., :3], what + ": accumulator against the oracle")
    assert_bit_equal(got["last"][..., :3], orc["last"][..., :3], what + ": last sample colour against the oracle")
    assert_bit_equal(got["rgba8"], orc["rgba8"][mode], what + ": rgba8 against the oracle")
    for g, r, name in zip(got["primary"], orc["primary"], ("index", "t", "count", "pos", "dir")):
        assert_bit_equal(g, r, "%s: primary %s against the oracle" % (what, name))
    assert got["counters"] == orc["counters"], (what, got["counters"], orc["counters"])


def _page_locked(a, keep):
    """A copy of `a` on pages of its own, page-locked (so that no two registered ranges share a page)."""
    page = 4096
    raw = np.empty(a.nbytes + 2 * page, np.uint8)
    off = (-raw.ctypes.data) % page
    b = raw[off:off + a.nbytes].view(a.dtype).reshape(a.shape)
    b[...] = a
    capi.host_register(b)
    keep.append((raw, b))
    return b


@gpu
@pytest.mark.parametrize("walk", list(WALKS))
def test_scene_walk_through_one_context(walk, monkeypatch):
    spec = WALKS[walk]
    steps = walk_scenes()
    for name in KNOB_NAMES:
        monkeypatch.delenv(name, raising=False)
    for i in range(len(steps)):  # the references first, with no knob set
        for mode in (0, 1):
            fresh_step(i, mode)
    locked, copies, uploads = [], {}, [sa for _, sa, _ in steps]
    if spec.get("pinned"):
        for i, sa in enumerate(uploads):
            uploads[i] = copy.copy(sa)
            for field in ("atlas", "env"):
                a = getattr(sa, field)
                if id(a) not in copies:
                    copies[id(a)] = _page_locked(a, locked)
                setattr(uploads[i], field, copies[id(a)])
    ctx = capi.Context(W, H)
    try:
        ctx.set_param(capi.PARAM_ANYHIT, 0)  # closest-hit traversal of every ray: node and leaf visits as in the oracle
        for i, (name, sa, _) in enumerate(steps):
            wait = spec["waits"][i % len(spec["waits"])]
            if spec.get("knobs"):
                for k in KNOB_NAMES:
                    monkeypatch.delenv(k, raising=False)
                for k, v in KNOBS[i % len(KNOBS)].items():
                    monkeypatch.setenv(k, v)
            if i == REFUSED_BEFORE:
                with pytest.raises(capi.FsptError) as e:
                    ctx.scene_upload(_refused(), wait=wait)
                assert e.value.code == E_LIMIT
                with pytest.raises(capi.FsptError) as e:
                    ctx.render(_frame(ctx, steps[i - 1][2]), 0, *_rand(i - 1))
                assert e.value.code == E_STATE, "a render after a refused upload"
            ctx.scene_upload(uploads[i], wait=wait)
            mode = (i + list(WALKS).index(walk)) % 2
            what = "%s walk, step %d (%s, %s, %s)" % (walk, i, name, "sum" if mode else "mean",
                                                     "wait" if wait else "no wait")
            if spec.get("knobs"):
                what += " %r" % (KNOBS[i % len(KNOBS)],)
            _check_step(_render_step(ctx, i, mode), i, mode, what)
    finally:
        try:
            ctx.synchronize()  # (an asynchronous upload may still read a page-locked atlas)
        finally:
            ctx.close()
            for _, b in locked:
                capi.host_unregister(b)


# ---------------------------------------------------------------------------------------------------------------------
# settings of the context apply to the scene after a swap
@gpu
def test_context_settings_survive_a_scene_swap():
    """Any-hit off, refraction cap 2, a tile and sum mode, all set before the swap, against a fresh context given the
    same settings (the tile's pixels: the oracle's sums; the others: untouched)."""
    import oracle
    first, second = walk_scenes()[_step("pbr_r32")], walk_scenes()[_step("dielectrics_r24")]  # both refractive
    x0, y0, w, h = 7, 5, 41, 30
    rc, rt = scenes.rand_bases(TICKS, 91)

    def run(ctx, before):
        ctx.set_param(capi.PARAM_ANYHIT, 0)
        ctx.set_param(capi.PARAM_MAX_REFRACTIONS, 2)
        ctx.set_tile(x0, y0, w, h)
        ctx.set_accum_mode(1)
        if before:
            ctx.scene_upload(first[1])
            ctx.render(_frame(ctx, first[2]), 0, rc, rt)
        ctx.scene_upload(second[1])
        ctx.clear()
        capped0 = ctx.stats()["capped_paths"]
        ctx.render(_frame(ctx, second[2]), 0, rc, rt)
        s = ctx.stats()
        return ctx.read_accum(), ctx.debug_last_color()[y0:y0 + h, x0:x0 + w], \
            (s["last_rays"], s["last_node_visits"], s["last_leaf_visits"], s["capped_paths"] - capped0)

    out = []
    for before in (True, False):
        ctx = capi.Context(W, H)
        try:
            out.append(run(ctx, before))
        finally:
            ctx.close()
    (acc, last, counters), (acc1, last1, counters1) = out
    assert_bit_equal(acc, acc1, "accumulator against a fresh context")
    assert_bit_equal(last, last1, "last sample colour against a fresh context")
    assert counters == counters1 and counters[3] > 0, (counters, counters1)
    sa, cam = second[1], second[2]
    O = oracle.Oracle(sa)
    ref = np.zeros((H, W, 4), np.float32)
    for k in range(TICKS):
        pos, d = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        col = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], max_refractions=2, want_color=True)[1]
        ref[y0:y0 + h, x0:x0 + w, :3] += col[y0:y0 + h, x0:x0 + w, :3]
    ref[y0:y0 + h, x0:x0 + w, 3] = TICKS
    assert_bit_equal(acc, ref, "sum accumulator of the tile against the oracle at refraction cap 2")


# ---------------------------------------------------------------------------------------------------------------------
# adaptive sampling: checkpoints, clear, swap
AW, AH, AN, BATCH, MIN_S = 64, 48, 16, 4, 4


def _adaptive_calls(ctx, fr, rc, rt, first_call=0):
    """Adaptive calls of BATCH ticks from call `first_call` on: [(active pixels before the call, accumulator, moment)]"""
    trail = []
    for k0 in range(first_call * BATCH, AN, BATCH):
        n = ctx.active_pixels()
        ctx.render(fr, k0, rc[k0:k0 + BATCH], rt[k0:k0 + BATCH])
        trail.append((n, ctx.read_accum(), ctx.read_moment()))
    return trail


def _assert_same_trail(got, ref, what):
    assert len(got) == len(ref)
    for c, ((n, acc, m2), (n1, acc1, m21)) in enumerate(zip(got, ref)):
        assert n == n1, "%s, call %d: active pixels %d, uninterrupted %d" % (what, c, n, n1)
        assert_bit_equal(acc, acc1, "%s, call %d: accumulator" % (what, c))
        assert_bit_equal(m2, m21, "%s, call %d: moment" % (what, c))


@pytest.fixture(scope="module")
def adaptive_case():
    """(scene, camera, rand bases, a threshold that stops some pixels at MIN_S and leaves others at AN)"""
    _, sa, cam = walk_scenes()[0]
    rc, rt = scenes.rand_bases(AN, 41)
    ctx = capi.Context(AW, AH)
    try:
        ctx.scene_upload(sa)
        accs, _, m2s = adaptive._uniform(ctx, _frame(ctx, cam), rc, rt)
    finally:
        ctx.close()
    err, _ = adaptive._pick_threshold(accs, m2s, adaptive._wave_starts(AN, BATCH, BATCH), MIN_S)
    return sa, cam, rc, rt, err


@gpu
def test_adaptive_checkpoint_continues_in_another_context(adaptive_case):
    """Accumulator + moment + next tick written into a second context (adaptive, sum mode) continue to the bits of the
    uninterrupted render, with the same active pixels before every call; the second checkpoint comes after pixels have
    stopped.  And fspt_clear followed by the same adaptive render gives the same bits again."""
    sa, cam, rc, rt, err = adaptive_case
    ctx = capi.Context(AW, AH)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        ctx.set_accum_mode(1)
        ctx.set_adaptive(err, MIN_S)
        ctx.clear()
        trail = _adaptive_calls(ctx, fr, rc, rt)
        last, samples = ctx.debug_last_color(), ctx.stats()["samples"]
        n_final = trail[-1][1][..., 3]
        assert n_final.min() < n_final.max() == AN
        ctx.clear()
        _assert_same_trail(_adaptive_calls(ctx, fr, rc, rt), trail, "adaptive render after fspt_clear")
        assert_bit_equal(ctx.debug_last_color(), last, "last sample colour after fspt_clear")
        assert ctx.stats()["samples"] == samples == int(n_final.sum())
    finally:
        ctx.close()
    for k in (1, 2):
        _, acc, m2 = trail[k - 1]
        if k == 2:
            assert (acc[..., 3] < k * BATCH).any(), "no pixel stopped before the checkpoint"
        ctx = capi.Context(AW, AH)
        try:
            ctx.scene_upload(sa)
            ctx.set_accum_mode(1)
            ctx.set_adaptive(err, MIN_S)
            ctx.write_accum(acc, k * BATCH)
            ctx.write_moment(m2)
            _assert_same_trail(_adaptive_calls(ctx, _frame(ctx, cam), rc, rt, first_call=k), trail[k:],
                               "continued after %d calls" % k)
            grown = n_final > acc[..., 3]
            assert_bit_equal(ctx.debug_last_color()[grown], last[grown], "last sample colour after %d calls" % k)
            assert ctx.stats()["samples"] == int(n_final.sum() - acc[..., 3].sum())
        finally:
            ctx.close()


@gpu
def test_adaptive_render_after_a_swap_and_clear_equals_a_fresh_context(adaptive_case):
    _, cam0, rc, rt, err = adaptive_case
    _, sa, cam = walk_scenes()[_step("pbr_r32")]
    out = []
    for swap in (True, False):
        ctx = capi.Context(AW, AH)
        try:
            ctx.set_accum_mode(1)
            ctx.set_adaptive(err, MIN_S)
            if swap:
                ctx.scene_upload(adaptive_case[0])
                _adaptive_calls(ctx, _frame(ctx, cam0), rc, rt)
            ctx.scene_upload(sa)
            ctx.clear()
            out.append((_adaptive_calls(ctx, _frame(ctx, cam), rc, rt), ctx.stats()["samples"]))
        finally:
            ctx.close()
    _assert_same_trail(out[0][0], out[1][0], "adaptive render after a swap")
    assert out[0][1] == out[1][1]


@gpu
def test_write_moment_before_adaptive_sampling_was_on():
    ctx = capi.Context(AW, AH)
    try:
        with pytest.raises(capi.FsptError) as e:
            ctx.write_moment(np.zeros((AH, AW), np.float32))
        assert e.value.code == E_STATE
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the walk covers what it claims
def _pow2(v):
    return v & (v - 1) == 0


def _dims(sa):
    p = capi.debug_pack_scene(sa)
    atlas = np.ascontiguousarray(sa.atlas)
    texels = atlas.view(np.uint32).reshape(atlas.shape[0], -1)
    constant = (texels == texels[:, :1]).all(axis=1)  # the host's constant-layer test: every texel equals the first
    quads = np.unique(np.asarray(sa.mats)[:, :4].astype(np.int64), axis=0)
    return dict(tris=sa.tris.shape[0], interior=p["n_interior"], depth=p["depth"], leaf_root=p["n_interior"] == 0,
                env_w=sa.env.shape[1], env_h=sa.env.shape[0], env_pow2=_pow2(sa.env.shape[1]) and _pow2(sa.env.shape[0]),
                bins=sa.bins.shape[0], res=atlas.shape[1], layers=atlas.shape[0],
                textured=int((~constant[quads].all(axis=1)).sum()), dielectric=p["dielectric"])


def _grow_shrink_grow(v):
    """Some step exceeds everything before it (storage re-made), a later one is smaller than its predecessor (storage
    kept), and a step after that exceeds everything before it again."""
    remade = [i for i in range(1, len(v)) if v[i] > max(v[:i])]
    shrunk = [i for i in range(1, len(v)) if v[i] < v[i - 1]]
    return any(a < s < b for a in remade for s in shrunk for b in remade)


def test_the_walk_covers_every_dimension():
    d = [_dims(sa) for _, sa, _ in walk_scenes()]
    pairs = list(zip(d, d[1:]))
    for key in ("tris", "interior"):
        assert _grow_shrink_grow([x[key] for x in d]), key
    assert any(a["leaf_root"] and b["depth"] == 64 for a, b in pairs), "a leaf root followed by a deep tree"
    assert any(a["depth"] == 64 and b["leaf_root"] for a, b in pairs), "a deep tree followed by a leaf root"
    for key in ("depth", "env_w", "env_h", "bins", "res", "layers"):  # (64 levels, the stack's limit, is the deepest)
        assert any(b[key] > a[key] for a, b in pairs) and any(b[key] < a[key] for a, b in pairs), key
    same_w = [(a, b) for a, b in pairs if a["env_w"] == b["env_w"]]
    assert any(b["env_h"] > a["env_h"] for a, b in same_w) and any(b["env_h"] < a["env_h"] for a, b in same_w), \
        "the environment's height alone changes, both ways"
    assert any(a["env_pow2"] and not b["env_pow2"] for a, b in pairs)
    assert any(not a["env_pow2"] and b["env_pow2"] for a, b in pairs)
    assert any(x["bins"] == 1 and x["env_w"] == x["env_h"] == 1 for x in d), "a 1-bin environment"
    same_r = [(a, b) for a, b in pairs if a["res"] == b["res"]]
    assert any(a["textured"] != b["textured"] for a, b in same_r), "textured materials change at the same resolution"
    assert any(a["textured"] != b["textured"] and a["layers"] == b["layers"] for a, b in same_r), \
        "textured materials change at the same resolution and layer count"
    assert any(a["textured"] == b["textured"] > 0 and a["tris"] != b["tris"] for a, b in same_r), \
        "another scene with the same interleaved atlas shape (the array is kept)"
    assert not d[0]["dielectric"]
    assert any(not a["dielectric"] and b["dielectric"] for a, b in pairs)
    assert any(a["dielectric"] and not b["dielectric"] for a, b in pairs)
    assert 0 < REFUSED_BEFORE < len(d)
    with pytest.raises(capi.FsptError) as e:
        capi.debug_pack_scene(_refused())
    assert e.value.code == E_LIMIT
