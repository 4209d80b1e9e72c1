"""The traversal against the CPU oracle, bit for bit, on scenes built to reach the kernel's edges: rays of more than 2^16
node and leaf visits (a flat fan, a soup of slivers through one point), subnormal and overflowed slab intermediates
(subnormal coordinates and origins, a mesh at 2^-126 .. 2^-140, a ground of +-1e30 and +-3e38), coincident box faces,
equal child distances and equal-t hits in different leaves (geometry at 2^20, every triangle twice), and the any-hit
exit of hit-or-miss rays.

The tests marked `gpu` compare k_trace's (index, t, count), its node / leaf visit counters and short renders with the
oracle, on both node-fetch paths; the others check, without a GPU, that each scene really reaches the edge it is about.
"""
import types

import numpy as np
import pytest

from fspt_b200 import capi, procedural as pr, scenes
import test_gpu_edges as edges  # degenerate_rays and the bit-equality helper

gpu = pytest.mark.gpu
F = np.float32
SUB = 2.0 ** -149  # the smallest subnormal
MAX_T, EPSILON = F(100000.0), F(0.000001)  # tracer.fs:10-11
LAST_BOUNCE = np.array([-2], np.int32).view(np.float32)[0]  # dir4.w marking a hit-or-miss ray (fspt_debug_trace)


def build(verts, camera):
    """A triangle soup (T, 3, 3) through the host builder and scene.flatten, with the camera its render uses."""
    verts = np.asarray(verts, np.float64).reshape(-1, 3, 3)
    p = dict(mesh=(verts.reshape(-1, 3), np.arange(verts.shape[0] * 3).reshape(-1, 3), None), scale=1, rotate=[],
             translate=[0, 0, 0], emittance=[0, 0, 0], normals="flat", diffuse=[0.8, 0.7, 0.6])
    sa = scenes.compile_props([p], {}, 4, scenes._env((64, 32)), builder=capi.bvh_build)
    return sa, dict(camera, fov_scale=0.5, env_theta=0.7, aperture=0.0, focal_depth=2.0)


def unit_mesh(seed):
    """An icosphere and a soup of mid-sized triangles, all within [-1.3, 1.3]^3"""
    v, f = pr.icosphere(2)
    return np.concatenate([v[f] * 0.5, pr.triangle_soup(600, seed, edge=(0.05, 0.3))])


def unit_dirs(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def rays(p, d):
    """(pos4, dir4) from (n, 3) origins and directions"""
    p, d = np.broadcast_arrays(np.asarray(p, F).reshape(-1, 3), np.asarray(d, F).reshape(-1, 3))
    pos, dir4 = np.ones((p.shape[0], 4), F), np.ones((p.shape[0], 4), F)
    pos[:, :3], dir4[:, :3] = p, d
    return pos, dir4


# ---------------------------------------------------------------------------------------------------------
# the scenes; each returns (scene arrays, camera, the (n, 3) origins and directions of the rays aimed at its edge)
def fan(T=600000):
    """T triangles sharing the centre vertex in the plane y = 0: a ray lying in that plane misses them all (det = 0) and
    enters every box it crosses (the y slab gives 0 * inf = NaN, ignored by min/max), ~2 x 10^5 visits, half leaves."""
    a = np.arange(T + 1) * (2 * np.pi / T)
    rim = np.c_[np.cos(a), np.zeros(T + 1), np.sin(a)]
    v = np.zeros((T, 3, 3))
    v[:, 1], v[:, 2] = rim[:-1], rim[1:]
    sa, cam = build(v, dict(eye=[0.1, 1.2, 1.6], dir=[-0.05, -0.6, -1.0]))
    p = np.array([[-2, 0, 0.001], [-2, 0, -0.3], [2, 0, 0.2], [0.001, 0, -2], [-1.5, 0, -1.5], [0.0, 0.0, 0.0]])
    d = np.array([[1, 0, 0], [1, 0, 0.01], [-1, 0, 0], [0, 0, 1], [1, 0, 1], [0.6, 0, 0.8]])
    rng = np.random.default_rng(31)
    q = rng.uniform(-1.5, 1.5, (64, 3))
    return sa, cam, (np.r_[p, q, q * [1, 0, 1]], np.r_[d, unit_dirs(rng, 64), unit_dirs(rng, 64) * [1, 0, 1]])


def slivers(T=140000):
    """T slivers p, -p, -p + 0.02 noise through the origin, p a random unit vector: every box holds the origin, so every
    ray from next to it visits every node (~10^5); depth 58 fits the 64-entry stack."""
    rng = np.random.default_rng(2)
    p = unit_dirs(rng, T)
    sa, cam = build(np.stack([p, -p, -p + 0.02 * rng.normal(size=(T, 3))], 1),
                    dict(eye=[1e-3, 1e-3, 1e-3], dir=[0.2, -0.3, -1.0]))
    return sa, cam, (np.full((48, 3), 1e-3), unit_dirs(rng, 48))


def subnormal():
    """Coordinates within 0.05 of 0 moved to +-k 2^-149: box faces at subnormal coordinates; rays start at 0 or at
    subnormal coordinates, so b - o and (b - o) / d are subnormal while triangles are still hit."""
    v = unit_mesh(41)
    rng = np.random.default_rng(41)
    small = np.abs(v) < 0.05
    v[small] = np.where(v[small] < 0, -1.0, 1.0) * rng.integers(1, 1024, int(small.sum())) * SUB
    sa, cam = build(v, dict(eye=[0.0, 0.0, 0.0], dir=[0.3, -0.2, -1.0]))
    n = 1024
    p = rng.integers(-64, 65, (n, 3)) * SUB * (rng.random((n, 3)) < 0.7)  # 0, +-0 or subnormal components
    d = unit_dirs(rng, n)
    d[: n // 4] *= rng.random((n // 4, 3)) < 0.6  # some axis-parallel (zero components)
    d[n // 4: n // 2, 0] = rng.integers(1, 64, n // 4) * SUB  # a subnormal component
    return sa, cam, (p, d)


def tiny():
    """The unit mesh at 2^-126, 2^-133 and 2^-140: every |det| falls below EPSILON, every ray misses, the visit counts
    alone decide."""
    v = unit_mesh(43)
    sa, cam = build(np.concatenate([v * 2.0 ** -126, v * 2.0 ** -133, v * 2.0 ** -140]),
                    dict(eye=[0.0, 0.0, 2.0], dir=[0.0, 0.0, -1.0]))
    rng = np.random.default_rng(43)
    n = 768
    p = rng.uniform(-1.5, 1.5, (n, 3)) * np.repeat([2.0 ** -126, 2.0 ** -133, 2.0 ** -140], n // 3)[:, None]
    return sa, cam, (p, unit_dirs(rng, n))


def ground():
    """The unit mesh over a quad of +-1e30 at y = -1 and one of +-3e38 at y = -2: e1 / e2 and det overflow (invDet = 0),
    and b - o overflows to +-inf for origins far out."""
    big = lambda y, s, x0=-1.0: np.array([[[x0 * s, y, -s], [s, y, s], [s, y, -s]], [[x0 * s, y, -s], [x0 * s, y, s], [s, y, s]]])  # noqa: E731
    v = np.concatenate([unit_mesh(47), big(-1.0, 1e30, 0.0), big(-2.0, 3e38)])
    sa, cam = build(v, dict(eye=[0.5, 2.0, 3.0], dir=[-0.2, -0.6, -1.0]))
    rng = np.random.default_rng(47)
    n = 512
    far = rng.choice([-3e38, -2e38, -1e38, 1e38, 2e38, 3e38, 1e30, -1e30], (n, 3))
    near = rng.uniform(-1.5, 1.5, (n, 3))
    pick = rng.random((n, 3)) < 0.5
    p = np.where(pick, far, near)
    d = near * 0.5 - p
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    q = np.c_[rng.uniform(-5e37, 5e37, (n, 2)), np.full(n, 3.0)][:, [0, 2, 1]]  # from above, onto the huge quads
    return sa, cam, (np.r_[p, q], np.r_[d, np.tile([[0.0, -1.0, 0.0]], (n, 1)) + rng.normal(0, 1e-3, (n, 3))])


def far_ties():
    """The unit mesh, every triangle twice, at about 2^20 (ulp 1/8): coincident box faces, equal child distances
    (lh == rh) and equal-t hits in different leaves."""
    v = unit_mesh(53) + 2.0 ** 20
    sa, cam = build(np.concatenate([v, v[::-1]]), dict(eye=[2 ** 20 + 0.3, 2 ** 20 + 1.5, 2 ** 20 + 3.0],
                                                         dir=[-0.1, -0.5, -1.0]))
    rng = np.random.default_rng(53)
    n = 1024
    p = 2.0 ** 20 + np.round(rng.uniform(-12, 12, (n, 3))) / 8  # on the 1/8 grid of the coordinates
    d = unit_dirs(rng, n)
    d[: n // 2] = np.eye(3)[rng.integers(0, 3, n // 2)] * rng.choice([-1, 1], (n // 2, 1))  # axis-parallel
    return sa, cam, (p, d)


SCENES = {"fan600k": fan, "slivers140k": slivers, "subnormal": subnormal, "tiny": tiny, "ground": ground,
          "far_ties": far_ties}
_built = {}


def scene(name):
    """sa, cam, oracle, edge = (pos4, dir4) of the scene's edge rays, rays = the degenerate-ray set of test_gpu_edges
    followed by the edge rays"""
    if name not in _built:
        import oracle
        sa, cam, (p, d) = SCENES[name]()
        pos, dir4 = edges.degenerate_rays(sa)
        ep, ed = rays(p, d)
        _built[name] = types.SimpleNamespace(sa=sa, cam=cam, oracle=oracle.Oracle(sa), edge=(ep, ed),
                                             rays=(np.r_[pos, ep], np.r_[dir4, ed]))
    return _built[name]


# ---------------------------------------------------------------------------------------------------------
# numpy restatements of the box and triangle arithmetic (tracer.fs:300-326) for the edge checks
def slab(box, o, inv, ftz=False):
    """rayBoxIntersect per (box, ray): boxes (B, 6), origins / inverse directions (R, 3) -> (B, R).  ftz: what a packed
    pipe that flushes subnormal inputs and results to zero would compute."""
    flush = (lambda a: np.where(np.abs(a) < F(2.0 ** -126), F(0.0) * np.sign(a), a)) if ftz else (lambda a: a)  # noqa: E731
    with np.errstate(all="ignore"):
        b, o, inv = flush(box[:, None, :]), flush(o[None]), flush(inv[None])
        t1 = flush(flush(b[..., :3] - o) * inv)
        t2 = flush(flush(b[..., 3:] - o) * inv)
    tmax = np.fmin(np.fmin(np.fmax(t1[..., 0], t2[..., 0]), np.fmax(t1[..., 1], t2[..., 1])), np.fmax(t1[..., 2], t2[..., 2]))
    tmin = np.fmax(np.fmax(np.fmin(t1[..., 0], t2[..., 0]), np.fmin(t1[..., 1], t2[..., 1])), np.fmin(t1[..., 2], t2[..., 2]))
    return np.where((tmax >= tmin) & (tmax > 0), tmin, MAX_T)


def boxes_and_rays(name):
    """the scene's node records, and the origins and inverse directions of its edge rays"""
    S = scene(name)
    pos, d = S.edge
    with np.errstate(divide="ignore", over="ignore"):
        inv = F(1.0) / d[:, :3]
    return np.ascontiguousarray(S.sa.bvh, F).reshape(-1, 9), pos[:, :3], inv


def interior(bvh):
    hdr = bvh.view(np.int32)
    i = np.flatnonzero(hdr[:, 2] < 0)
    return hdr[i, 0], hdr[i, 1]


# ---------------------------------------------------------------------------------------------------------
# CPU: each scene reaches its edge
@pytest.mark.parametrize("name", list(SCENES))
def test_scene_fits_the_stack_and_any_hit_agrees_with_closest_hit(name):
    S = scene(name)
    sa, O, (pos, d) = S.sa, S.oracle, S.rays
    assert capi.debug_pack_scene(sa)["depth"] <= 64  # the upload's own depth check: levels, root included
    ci, ct, cc, cst = O.bvh_test(pos, d)
    ai, at, ac, ast = O.bvh_test(pos, d, anyhit=True)
    assert cst["stack_overflow"] == 0 and ast["stack_overflow"] == 0
    assert ((ai >= 0) == (ci >= 0)).all() and (ac <= cc).all()
    assert (at[ai < 0] == MAX_T).all() and (at[ai >= 0] >= ct[ai >= 0]).all()
    hits = ci >= 0
    if name != "tiny":
        assert hits.sum() > 10 and (ac[hits] < cc[hits]).any()  # the exit is taken


def test_fan_and_slivers_pass_two_to_the_16_visits():
    import oracle
    S = scene("fan600k")
    pos, d = S.edge
    _, _, c1, s1 = S.oracle.bvh_test(pos[:1], d[:1])  # one ray alone: its own leaf visits
    assert c1[0] > 2 * 65536 and s1["leaf_visits"] > 65536 and s1["node_visits"] - s1["leaf_visits"] > 65536
    _, _, cnt, _ = S.oracle.bvh_test(pos, d)
    assert (cnt > 65536).sum() >= 4
    S = scene("slivers140k")
    _, _, cnt, _ = S.oracle.bvh_test(*S.edge)
    assert (cnt > 65536).all()
    cam = S.cam
    cp, cd = oracle.camera(*SIZE, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), F(17.0))
    _, _, cnt, st = S.oracle.bvh_test(cp, cd)
    assert (cnt > 65536).all() and st["leaf_visits"] > 65536 * cnt.size // 2  # every camera ray of the render


def test_subnormal_intermediates_decide_box_tests():
    bvh, o, inv = boxes_and_rays("subnormal")
    box = bvh[:, 3:9]
    with np.errstate(all="ignore"):
        diff = box[:, None, :3] - o[None]
        prod = diff * inv[None]
    sub = lambda a: (a != 0) & (np.abs(a) < F(2.0 ** -126))  # noqa: E731
    assert sub(box).any() and sub(o).any() and sub(diff).any() and sub(prod).any()
    exact, ftz = slab(box, o, inv), slab(box, o, inv, ftz=True)
    assert (bits(exact) != bits(ftz)).sum() > 100  # flushing them would change box hits and entry distances
    S = scene("subnormal")
    idx, _, _, _ = S.oracle.bvh_test(*S.edge)
    assert (idx >= 0).sum() > 100


def test_tiny_mesh_is_all_misses():
    S = scene("tiny")
    tris = np.ascontiguousarray(S.sa.tris, F).reshape(-1, 3, 3)
    assert (np.abs(tris) < F(2.0 ** -120)).all() and (tris != 0).any()
    idx, _, _, _ = S.oracle.bvh_test(*S.rays)
    _, _, cnt, _ = S.oracle.bvh_test(*S.edge)
    assert (idx < 0).all() and (cnt > 8).sum() > 200
    bi, _ = S.oracle.brute_force(*S.edge)
    assert (bi < 0).all()


def test_ground_overflows():
    S = scene("ground")
    tris = np.ascontiguousarray(S.sa.tris, F).reshape(-1, 3, 3)
    with np.errstate(over="ignore"):
        e1 = tris[:, 1] - tris[:, 0]
    assert np.isinf(e1).any()  # det = dot(e1, cross(d, e2)) overflows too, invDet = 0
    bvh, o, inv = boxes_and_rays("ground")
    with np.errstate(over="ignore", invalid="ignore"):
        diff = bvh[:, None, 3:6] - o[None]
    assert np.isinf(diff).any()
    idx, _, _, _ = S.oracle.bvh_test(*S.rays)
    big = np.flatnonzero(np.abs(tris).max(axis=(1, 2)) > 1e29)
    aimed = S.oracle.bvh_test(*S.edge)[0][-512:]  # the rays from above onto the quads
    # det = dot(e1, cross(d, e2)) overflows, invDet = 0, dist = 0: the huge quads are never hit, the mesh still is
    assert not np.isin(idx, big).any() and (aimed == -1).sum() > 100 and (idx >= 0).sum() > 50


def test_far_scene_has_ties():
    bvh, o, inv = boxes_and_rays("far_ties")
    L, R = interior(bvh)
    lh, rh = slab(bvh[L, 3:9], o, inv), slab(bvh[R, 3:9], o, inv)
    assert ((lh == rh) & (lh < MAX_T)).sum() > 100  # equal child distances: the tie goes left
    assert (bvh[L, 3:9] == bvh[R, 3:9]).any(axis=1).sum() > 100  # coincident faces
    S = scene("far_ties")
    idx, _, _, _ = S.oracle.bvh_test(*S.rays)
    tris = np.ascontiguousarray(S.sa.tris, F).reshape(-1, 9)
    first = np.sort(bvh.view(np.int32)[:, 2][bvh.view(np.int32)[:, 2] >= 0])
    leaf = lambda i: first[np.searchsorted(first, i, side="right") - 1]  # noqa: E731
    _, inv_u, cnt_u = np.unique(tris.view(np.uint32), axis=0, return_inverse=True, return_counts=True)
    inv_u = inv_u.ravel()
    ties = 0
    for i in idx[idx >= 0]:
        twins = np.flatnonzero(inv_u == inv_u[i])
        ties += any(leaf(j) != leaf(i) for j in twins if j != i)  # the same t from a triangle of another leaf
    assert (cnt_u == 2).all() and ties > 20


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


# ---------------------------------------------------------------------------------------------------------
# GPU: k_trace against the oracle
SIZE = (24, 16)


def _oracle_render(O, cam, rc, rt):
    """tracer.fs over len(rc) ticks: accumulator, the last tick's per-sample colours, summed stats"""
    import oracle
    W, H = SIZE
    fb, tot = None, {}
    for k in range(len(rc)):
        pos, d = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        fb, col, st = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fb, want_color=True)
        tot = {key: tot.get(key, 0) + v for key, v in st.items()}
    return fb, col, tot


_renders, _traces = {}, {}  # oracle results, shared by the two node-fetch paths


@gpu
@pytest.mark.parametrize("node_tex", [True, False], ids=["node_tex", "lsu"])
@pytest.mark.parametrize("name", list(SCENES))
def test_traversal_edges(name, node_tex, monkeypatch):
    """(index, t, count) closest-hit and any-hit, the visit counters over those traces, and a short render with
    ANYHIT 0 and 1 (accumulator, last colour, rays, and at ANYHIT 0 the visit counters), all equal to the oracle's."""
    if not node_tex:
        monkeypatch.setenv("FSPT_NO_NODE_TEX", "1")
    S = scene(name)
    sa, cam, O, (pos, d) = S.sa, S.cam, S.oracle, S.rays
    ctx = capi.Context(*SIZE)
    try:
        ctx.scene_upload(sa)
        for anyhit_param in (1, 0):
            ctx.set_param(capi.PARAM_ANYHIT, anyhit_param)
            for marked in (False, True):
                dm = d.copy()
                if marked:
                    dm[:, 3] = LAST_BOUNCE
                what = "%s, %s ray, ANYHIT %d" % (name, "hit-or-miss" if marked else "closest-hit", anyhit_param)
                before = ctx.stats()
                idx, t, cnt = ctx.debug_trace(pos, dm)
                after = ctx.stats()
                key = (name, marked and anyhit_param == 1)
                if key not in _traces:
                    _traces[key] = O.bvh_test(pos, dm, anyhit=key[1])
                oi, ot, oc, st = _traces[key]
                edges.assert_bit_equal(idx, oi, "hit index, " + what)
                edges.assert_bit_equal(t, ot, "hit t, " + what)
                edges.assert_bit_equal(cnt, oc, "visit count, " + what)
                assert after["node_visits"] - before["node_visits"] == st["node_visits"], what
                assert after["leaf_visits"] - before["leaf_visits"] == st["leaf_visits"], what
        rc, rt = scenes.rand_bases(2, 97)
        if name not in _renders:
            _renders[name] = _oracle_render(O, cam, rc, rt)
        ofb, ocol, ost = _renders[name]
        fr = ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])
        for anyhit_param in (0, 1):
            ctx.set_param(capi.PARAM_ANYHIT, anyhit_param)
            ctx.clear()
            ctx.render(fr, 0, rc, rt)
            what = "%s, ANYHIT %d" % (name, anyhit_param)
            edges.assert_bit_equal(ctx.read_accum()[..., :3], ofb[..., :3], "accumulator, " + what)
            edges.assert_bit_equal(ctx.debug_last_color()[..., :3], ocol[..., :3], "last colour, " + what)
            s = ctx.stats()
            assert s["last_rays"] == ost["rays"], what
            if anyhit_param == 0:
                assert (s["last_node_visits"], s["last_leaf_visits"]) == (ost["node_visits"], ost["leaf_visits"]), what
            else:
                assert s["last_node_visits"] <= ost["node_visits"] and s["last_leaf_visits"] <= ost["leaf_visits"], what
    finally:
        ctx.close()
