"""The host half of fspt_scene_upload without a GPU (fspt_debug_pack_scene, fspt_b200/csrc/scene_pack.h): the device
records it builds -- Node64, Tri48, ShadeRec, material ids -- against a numpy restatement of the layouts from the
reference-format arrays (main.js:360-392), for any number of worker threads, and its error reports."""
import types

import numpy as np
import pytest

from fspt_b200 import capi, scenes


def _expected(sa):
    bvh = np.ascontiguousarray(sa.bvh, np.float32).reshape(-1, 9)
    hdr = bvh.view(np.int32)
    N, T = bvh.shape[0], sa.tris.shape[0]
    leaf = hdr[:, 2] > -1                                   # `current.triangles > -1`, tracer.fs:379
    ref = np.where(leaf, ~hdr[:, 2], np.cumsum(~leaf) - 1).astype(np.int32)
    interior = np.nonzero(~leaf)[0]
    node64 = np.zeros((len(interior), 16), np.float32)
    l, r = hdr[interior, 0], hdr[interior, 1]
    node64[:, 0:12:2] = bvh[l, 3:9]                         # (left, right) pairs per component: min xyz, max xyz
    node64[:, 1:12:2] = bvh[r, 3:9]
    node64.view(np.int32)[:, 12] = ref[l]
    node64.view(np.int32)[:, 13] = ref[r]
    tris = np.ascontiguousarray(sa.tris, np.float32).reshape(-1, 9)
    tri48 = np.zeros((T + 3, 12), np.float32)
    tri48[:T, 0:3] = tris[:, 0:3]
    tri48[:T, 3:6] = tris[:, 3:6] - tris[:, 0:3]            # f32 subtractions, tracer.fs:301-302
    tri48[:T, 6:9] = tris[:, 6:9] - tris[:, 0:3]
    tri48[T:, 0:3] = -1.0                                   # padBuffer's -1 fill: v = -1, e = (-1) - (-1) = 0
    mats = np.ascontiguousarray(sa.mats, np.float32).reshape(-1, 12)
    L = sa.atlas.shape[0]

    def layer(col):
        return np.clip(np.floor(col + np.float32(0.5)), 0, L - 1).astype(np.int64)
    keys = np.stack([layer(mats[:, 0]), layer(mats[:, 1]), layer(mats[:, 3]), layer(mats[:, 2])], 1)
    ids, mat_id = {}, np.zeros(T, np.int32)
    for t in range(T):                                       # order of first appearance
        mat_id[t] = ids.setdefault(tuple(keys[t]), len(ids))
    shaderec = np.zeros((T, 48), np.float32)
    shaderec[:, 0:12] = mats
    shaderec[:, 12:18] = np.ascontiguousarray(sa.uvs, np.float32).reshape(-1, 6)
    shaderec.view(np.int32)[:, 18] = mat_id
    shaderec[:, 20:47] = np.ascontiguousarray(sa.norms, np.float32).reshape(-1, 27)
    return dict(node64=node64, tri48=tri48, shaderec=shaderec, mat_id=mat_id, root_ref=int(ref[0]), n_materials=len(ids),
                dielectric=bool((mats[:, 10] >= 0).any()))


def _same(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("scene", ["bunny", "pbr", "quad", "soup"])
@pytest.mark.parametrize("threads", [1, 3, 16])
def test_device_records_match_the_reference_layout(scene, threads):
    if scene == "bunny":
        sa, _ = scenes.bunny_class(subdiv=4, atlas_res=16, env_size=(64, 32))
    elif scene == "pbr":
        sa, _ = scenes.pbr_scene(atlas_res=16, subdiv=3, env_size=(64, 32))      # several materials, one dielectric
    elif scene == "quad":
        sa, _ = scenes.quad_scene()                                              # the root is a leaf: no interior record
    else:
        sa, _ = scenes.sphere_soup(subdiv=3, n_soup=30000, env_size=(64, 32))    # > 8192 nodes / triangles: several chunks
    got, exp = capi.debug_pack_scene(sa, n_threads=threads), _expected(sa)
    assert got["n_interior"] == exp["node64"].shape[0] and got["root_ref"] == exp["root_ref"]
    if got["n_interior"]:
        assert _same(got["node64"], exp["node64"])
    assert _same(got["tri48"], exp["tri48"])
    assert _same(got["shaderec"], exp["shaderec"])
    assert np.array_equal(got["mat_id"], exp["mat_id"]) and got["n_materials"] == exp["n_materials"]
    assert got["dielectric"] == exp["dielectric"]
    assert got["depth"] == sa.depth + 1                     # nodes on the longest root-to-leaf path (the builder counts edges)


def test_material_ids_merge_across_chunks_in_order_of_first_appearance():
    """More than one pre-pass chunk (8192 triangles) with materials that first appear in different chunks, in an order
    that differs from the chunk-local numbering."""
    sa, _ = scenes.sphere_soup(subdiv=3, n_soup=30000, env_size=(64, 32))
    sa.mats = np.array(sa.mats, np.float32, copy=True)
    T = sa.mats.shape[0]
    layers = np.zeros((T, 4), np.float32)
    layers[T // 3:, 0] = 2          # second material from the middle of the scene on
    layers[2 * T // 3:, 1] = 1      # third one in the last chunk(s)
    layers[100:200, 0] = 2          # ... but the second one already shows up early, inside the first chunk
    sa.mats[:, 0:4] = layers
    sa.atlas = np.zeros((3, 4, 4, 4), np.uint8)
    got, exp = capi.debug_pack_scene(sa, n_threads=8), _expected(sa)
    assert got["n_materials"] == exp["n_materials"] == 3
    assert np.array_equal(got["mat_id"], exp["mat_id"])


def _chain(n, sa):
    bvh = np.zeros((2 * n + 1, 9), np.float32)
    hdr = bvh.view(np.int32)
    for i in range(n):
        hdr[2 * i, 0], hdr[2 * i, 1], hdr[2 * i, 2] = 2 * i + 1, 2 * i + 2, -1
        hdr[2 * i + 1, 2] = 0
    hdr[2 * n, 2] = 0
    bvh[:, 3:6], bvh[:, 6:9] = -1.0, 1.0
    return types.SimpleNamespace(bvh=bvh, tris=sa.tris[:4], mats=sa.mats[:4], norms=sa.norms[:4], uvs=sa.uvs[:4],
                                 atlas=sa.atlas, env=sa.env, bins=sa.bins, leaf_size=4)


def test_error_reports_of_the_pre_passes():
    sa, _ = scenes.bunny_class(subdiv=2, atlas_res=16, env_size=(64, 32))
    ok = capi.debug_pack_scene(_chain(63, sa))               # 64 levels: the sentinel + 63 deferred children fill the
    assert ok["depth"] == 64 and ok["n_interior"] == 63      # reference's int stack[64] (tracer.fs:368) exactly
    with pytest.raises(capi.FsptError) as e:                 # 65 levels: one deferred child more than the stack holds
        capi.debug_pack_scene(_chain(64, sa))
    assert e.value.code == -4 and "stack" in str(e.value) and "65 levels" in str(e.value)
    cyc = _chain(3, sa)
    cyc.bvh = cyc.bvh.copy()
    cyc.bvh.view(np.int32)[4, 0] = 0                         # an interior node points back at the root
    with pytest.raises(capi.FsptError) as e:
        capi.debug_pack_scene(cyc)
    assert e.value.code == -1 and ("tree" in str(e.value) or "child" in str(e.value))
    bad = _chain(3, sa)
    bad.bvh = bad.bvh.copy()
    bad.bvh.view(np.int32)[1, 2] = 4                         # leaf whose first triangle lies beyond the 4 triangles
    with pytest.raises(capi.FsptError) as e:
        capi.debug_pack_scene(bad)
    assert e.value.code == -1 and "triangle index" in str(e.value)
    oob = _chain(3, sa)
    oob.bvh = oob.bvh.copy()
    oob.bvh.view(np.int32)[2, 1] = 99                        # child index out of range
    with pytest.raises(capi.FsptError) as e:
        capi.debug_pack_scene(oob)
    assert e.value.code == -1 and "child index" in str(e.value)
