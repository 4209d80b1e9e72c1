"""fspt_bvh_build_device (csrc/bvh_device.cu) against the host builder (csrc/bvh_builder.cpp, pinned to bvh.js and to the
oracle): node records, leaf order, node count and depth bit for bit, the same refusals with the same codes, and the
choice between the two builders that scene.flatten makes."""
import numpy as np
import pytest

from fspt_b200 import capi, procedural as pr, scene, scenes
from fspt_b200.geometry import mesh_to_triangles

gpu = pytest.mark.gpu

# the device builder's internal cutoffs (csrc/bvh_device.cu): one-thread segments, block tile (radix, scans, chunks)
SMALL, TILE = 64, 2048


def no_gpu():
    import torch
    return not torch.cuda.is_available()


def assert_same_tree(verts, max_tris=4, box_verts=None):
    hn, ho, hd = capi.bvh_build(verts, max_tris, box_verts=box_verts)
    dn, do, dd = capi.bvh_build_device(verts, max_tris, box_verts=box_verts)
    assert dn.shape == hn.shape, "n_nodes %d vs host %d" % (dn.shape[0], hn.shape[0])
    assert np.array_equal(dn.view(np.uint32), hn.view(np.uint32)), "node records differ"
    assert np.array_equal(do, ho), "order differs"
    assert dd == hd, "depth %d vs host %d" % (dd, hd)
    return dn, do, dd


def _grid(n):
    """2 n^2 axis-aligned right triangles: every centroid coordinate ties with many others"""
    g = np.stack(np.meshgrid(np.arange(float(n)), np.arange(float(n)), indexing="ij"), -1).reshape(-1, 2)
    tri = np.zeros((len(g) * 2, 3, 3))
    tri[0::2, :, 0] = g[:, None, 0] + np.array([0, 1, 0]); tri[0::2, :, 1] = g[:, None, 1] + np.array([0, 0, 1])
    tri[1::2, :, 0] = g[:, None, 0] + np.array([1, 1, 0]); tri[1::2, :, 1] = g[:, None, 1] + np.array([0, 1, 1])
    return tri


def _meshes():
    """The inputs the bvh.js pin uses (tests/test_reference_js_pin.py)."""
    rng = np.random.default_rng(7)
    v2, f2 = pr.icosphere(2)
    v3, f3 = pr.icosphere(3)
    soup = rng.uniform(-1, 1, (1500, 1, 3)) + rng.normal(0, 0.05, (1500, 3, 3))
    grid = _grid(14)
    return {
        "quad_root_leaf": (pr.QUAD_VERTS[np.asarray(pr.QUAD_FACES)], None),
        "five_triangles": (soup[:5], None),
        "icosphere_lumpy": (pr.lumpy(v2)[f2], None),
        "icosphere_symmetric_ties": (v3[f3], None),
        "soup": (soup, None),
        "grid_all_ties": (grid, None),
        "stale_boxes_after_normalize": (grid * 0.37 + 0.1, grid),
        "duplicates": (np.concatenate([soup[:40], soup[:40]]), None),
        "four_point_triangles_one_leaf": (np.zeros((4, 3, 3)), None),
    }


def _soup(T, seed=11):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1, 1, (T, 1, 3)) + rng.normal(0, 0.02, (T, 3, 3))


def _tie_heavy(T, seed=5):
    """coordinates on a 1/32 grid and every fifth triangle a copy: equal centroids and equal SAH costs are common"""
    rng = np.random.default_rng(seed)
    c = np.round(rng.uniform(-1, 1, (T, 1, 3)) * 32) / 32
    v = (c + np.round(rng.uniform(-0.1, 0.1, (T, 3, 3)) * 32) / 32).reshape(-1, 9)
    v[1::5] = v[0::5][:v[1::5].shape[0]]
    return v


@gpu
@pytest.mark.parametrize("name", list(_meshes()))
def test_device_builder_matches_host_on_the_bvh_js_pin_inputs(name):
    verts, box = _meshes()[name]
    assert_same_tree(verts, 4, box)


@gpu
@pytest.mark.parametrize("leaf", [1, 2, 8])
def test_device_builder_other_leaf_sizes(leaf):
    verts, _ = _meshes()["icosphere_lumpy"]
    assert_same_tree(verts, leaf)
    assert_same_tree(_tie_heavy(5000), leaf)


@gpu
def test_device_builder_leaf_size_above_the_small_segment_size():
    assert_same_tree(_soup(3000), SMALL + 36)


@gpu
def test_device_builder_large_tie_heavy_input():
    assert_same_tree(_tie_heavy(140000))


@gpu
@pytest.mark.parametrize("T", [1, 2, 3, 5, SMALL - 1, SMALL, SMALL + 1, 2 * SMALL + 1, TILE - 1, TILE, TILE + 1, 2 * TILE + 1,
                               256 * TILE + 1, (1 << 17) - 1, 1 << 17, (1 << 17) + 1])
def test_device_builder_sizes_around_its_cutoffs(T):
    assert_same_tree(_soup(T, seed=T))
    assert_same_tree(_tie_heavy(T, seed=T))


@gpu
def test_device_builder_signed_zeros():
    """-0.0 and +0.0 centroids tie in the host's presort (`<`); box bounds keep Math.min/max's signed-zero rule."""
    rng = np.random.default_rng(3)
    T = 6000
    v = rng.uniform(-1, 1, (T, 3, 3))
    # x centroid (mn + mx) * 0.5 is -0.0 for a third, +0.0 for a third
    v[0::3, :, 0] = np.array([-0.0, -0.0, -0.0])
    v[1::3, :, 0] = np.array([0.0, 0.0, 0.0])
    # box bounds that are -0.0 / +0.0 on y and z, mixed within one triangle
    v[2::6, :, 1] = np.array([-0.0, 0.0, -0.0])
    v[5::6, :, 2] = np.array([0.0, -0.0, 0.5])
    assert np.signbit(v[0::3, :, 0]).all() and not np.signbit(v[1::3, :, 0]).any()
    assert_same_tree(v)
    assert_same_tree(v.copy(), 4, v * -1.0)


@gpu
def test_device_builder_config3_vertices():
    v = scenes.sphere_soup_verts()
    assert v.shape[0] == 1000000
    assert_same_tree(v)


@gpu
def test_device_builder_config5_vertices():
    v = scenes.sphere_soup_verts(subdiv=8, n_soup=10000000 - 1310720, seed=4321)
    assert v.shape[0] == 10000000
    assert_same_tree(v)


@gpu
@pytest.mark.parametrize("verts", [np.zeros((8, 3, 3)), np.ones((5, 3, 3)),
                                   np.concatenate([np.random.default_rng(1).normal(size=(40, 3, 3)), np.zeros((8, 3, 3))]),
                                   np.concatenate([np.zeros((3000, 3, 3)), _soup(200)])],
                         ids=["zeros", "one_point", "soup_plus_zeros", "many_zeros_plus_soup"])
def test_device_builder_refuses_where_the_host_refuses(verts):
    with pytest.raises(capi.FsptError) as host:
        capi.bvh_build(verts, 4)
    with pytest.raises(capi.FsptError) as dev:
        capi.bvh_build_device(verts, 4)
    assert dev.value.code == host.value.code == -4


@gpu
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
@pytest.mark.parametrize("where", ["verts", "box_verts"])
def test_device_builder_refuses_non_finite_vertices(bad, where):
    v = _soup(5000)
    box = v * 2.0
    (v if where == "verts" else box)[4321, 1, 2] = bad
    with pytest.raises(capi.FsptError) as host:
        capi.bvh_build(v, 4, box_verts=box)
    with pytest.raises(capi.FsptError) as dev:
        capi.bvh_build_device(v, 4, box_verts=box)
    assert dev.value.code == host.value.code == -1


@gpu
def test_device_builder_repeats_itself():
    v = _tie_heavy(300000, seed=9)
    first = capi.bvh_build_device(v)
    for _ in range(2):
        again = capi.bvh_build_device(v)
        assert np.array_equal(again[0].view(np.uint32), first[0].view(np.uint32))
        assert np.array_equal(again[1], first[1]) and again[2] == first[2]


@gpu
def test_device_build_between_renders_of_a_live_context(oracle_mod, small_bunny):
    """A build on the device of a live context neither synchronises nor disturbs it: the render after it stays bit-exact."""
    sa, cam = small_bunny
    W, H, N = 96, 64, 2
    ctx = capi.Context(W, H, 0)
    try:
        ctx.scene_upload(sa)
        fr = ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])
        rc, rt = scenes.rand_bases(N, 3)
        ctx.render(fr, 0, rc[:1], rt[:1])
        assert_same_tree(_soup(200000))
        ctx.render(fr, 1, rc[1:], rt[1:])
        fb = ctx.read_accum()
    finally:
        ctx.close()
    O = oracle_mod.Oracle(sa)
    ofb = None
    for k in range(N):
        pos, d = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        ofb, _ = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=ofb)
    assert np.array_equal(fb[..., :3].view(np.uint32), ofb[..., :3].view(np.uint32))


def _sets(T):
    p = dict(scale=1, rotate=[], translate=[0, 0, 0], emittance=[0, 0, 0], normals="flat", diffuse=[0.5, 0.5, 0.5])
    sv = _soup(T, seed=2).reshape(-1, 3)
    ts = mesh_to_triangles(sv, np.arange(sv.shape[0]).reshape(-1, 3), p)
    ts.material = dict(diffuseIndex=0, roughnessIndex=0, normalIndex=0, specularIndex=0, ior=1.4, dielectric=-1,
                       emittance=[0, 0, 0])
    return [ts]


def _flatten(T):
    return scene.flatten(_sets(T), np.zeros((1, 4, 4, 4), np.uint8), np.zeros((2, 4, 4), np.uint8),
                         np.array([[0, 0, 4, 2]], np.uint16))


@gpu
def test_flatten_builds_large_scenes_on_the_device(monkeypatch):
    calls = []
    for name in ("bvh_build", "bvh_build_device"):
        real = getattr(capi, name)
        monkeypatch.setattr(capi, name, lambda *a, _r=real, _n=name, **k: calls.append(_n) or _r(*a, **k))
    T = scene.DEVICE_BVH_MIN_TRIS
    big = _flatten(T)
    assert calls == ["bvh_build_device"]
    small = _flatten(T - 1)
    assert calls == ["bvh_build_device", "bvh_build"]
    ref = capi.bvh_build(_sets(T)[0].verts, 4)
    assert np.array_equal(big.bvh.view(np.uint32), ref[0].view(np.uint32)) and np.array_equal(big.order, ref[1])
    assert small.n_tris == T - 1


def test_device_builder_without_a_device_fails_loudly():
    if not no_gpu():
        pytest.skip("GPU present")
    with pytest.raises(capi.FsptError) as e:
        capi.bvh_build_device(_soup(100))
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)
    assert not capi.device_usable(0)


def test_flatten_without_a_builder_returns_the_host_builders_arrays():
    for T in (1000, scene.DEVICE_BVH_MIN_TRIS):
        sa = _flatten(T)
        nodes, order, depth = capi.bvh_build(_sets(T)[0].verts, 4)
        assert np.array_equal(sa.bvh.view(np.uint32), nodes.view(np.uint32))
        assert np.array_equal(sa.order, order) and sa.depth == depth
