"""Scene compilation: what main.js initBVH() does between parsing props and the texImage uploads
(main.js:284-445) -- materials -> atlas layers, BVH build, the flatten loop, environment + radiance bins --
producing the exact flattened arrays the reference uploads (SURVEY.md appendix A), ready for
fspt_scene_upload.  Host-side only; BVH construction and env bins run in the native library."""
import functools
from dataclasses import dataclass, field

import numpy as np

from . import capi
from .geometry import TriangleSet
from .texture_packer import TexturePacker


@dataclass
class SceneArrays:
    bvh: np.ndarray      # (N,9) f32, [0..2] int32 bits            main.js:366-392,272-282
    tris: np.ndarray     # (T,9) f32, leaf order                   main.js:374
    mats: np.ndarray     # (T,12) f32                              main.js:377-382
    norms: np.ndarray    # (T,27) f32                              main.js:383-385
    uvs: np.ndarray      # (T,6) f32                               main.js:386
    atlas: np.ndarray    # (L,res,res,4) u8                        main.js:556-559
    env: np.ndarray      # (H,W,4) u8 RGBE, row 0 = top            main.js:170-180
    bins: np.ndarray     # (B,4) u16                               main.js:298-299
    lights: np.ndarray = None        # (Lt,9) f32, unused by tracer.fs main()
    light_ranges: np.ndarray = None
    leaf_size: int = 4
    depth: int = 0
    order: np.ndarray = None         # source triangle of each triTex slot
    verts64: np.ndarray = None       # (T,9) f64 Triangle.verts in leaf order: what shootAutoFocusRay walks (main.js:447-546)

    @property
    def n_tris(self):
        return self.tris.shape[0]

    def nbytes(self):
        return sum(a.nbytes for a in (self.bvh, self.tris, self.mats, self.norms, self.uvs, self.atlas, self.env, self.bins))


def get_material(prop, group_material, packer, assets, base_path=""):
    """getMaterial (main.js:206-270).  `assets` maps url -> image dict.  Returns the material record."""
    gm = group_material or {}

    _keep = object()

    def tex(url, corrected=False, swizzle=_keep):
        # one mutable record per url, like the reference's Image elements: `img.swizzle = ...` is assigned on the
        # shared object for metallic-roughness maps only (main.js:228-229,235-236, `undefined` included) and is read
        # when the atlas is packed, so the LAST assignment wins for every layer made from that image
        img = assets[url]
        if swizzle is not _keep:
            img["swizzle"] = swizzle
        return packer.addTexture(img, corrected)

    if gm.get("map_kd"):
        diffuse = tex(base_path + "/" + gm["map_kd"], True)
    elif gm.get("kd"):
        diffuse = packer.addColor(gm["kd"])
    elif isinstance(prop.get("diffuse"), str):
        diffuse = tex(prop["diffuse"], True)
    elif isinstance(prop.get("diffuse"), (list, tuple)):
        diffuse = packer.addColor(prop["diffuse"])
    else:
        diffuse = packer.addColor([0.5, 0.5, 0.5])

    if gm.get("map_pmr"):
        rough = tex(base_path + "/" + gm["map_pmr"], None, gm.get("pmr_swizzle"))  # addTexture(img): corrected = undefined
    elif gm.get("pmr"):
        rough = packer.addColor(gm["pmr"])
    elif isinstance(prop.get("metallicRoughness"), str):
        rough = tex(prop["metallicRoughness"], None, prop.get("mrSwizzle"))
    elif isinstance(prop.get("metallicRoughness"), (list, tuple)):
        rough = packer.addColor(prop["metallicRoughness"])
    else:
        rough = packer.addColor([0.0, 0.3, 0])

    if gm.get("map_kem"):
        spec = tex(base_path + "/" + gm["map_kem"])
    elif gm.get("kem"):
        spec = packer.addColor(gm["kem"])
    elif isinstance(prop.get("emission"), str):
        spec = tex(prop["emission"])
    else:
        spec = packer.addColor([0, 0, 0])

    if gm.get("map_bump"):
        normal = tex(base_path + "/" + gm["map_bump"])
    elif prop.get("normal"):
        normal = tex(prop["normal"])
    else:
        normal = packer.addColor([0.5, 0.5, 1])

    def js_or(*vals):  # a || b || c
        for v in vals[:-1]:
            if v:
                return v
        return vals[-1]

    return {
        "diffuseIndex": diffuse, "roughnessIndex": rough, "normalIndex": normal, "specularIndex": spec,
        "ior": float(js_or(gm.get("ior"), prop.get("ior"), 1.4)),                    # main.js:266
        "dielectric": float(js_or(gm.get("dielectric"), prop.get("dielectric"), -1)),  # main.js:267
        "emittance": [float(x) for x in prop["emittance"]],                          # main.js:268 (required key)
    }


def material_row(m):
    """One materialBuffer record (main.js:377-382)."""
    return np.array([m["diffuseIndex"], m["specularIndex"], m["normalIndex"], m["roughnessIndex"], 0, 0,
                     m["emittance"][0], m["emittance"][1], m["emittance"][2], m["ior"], m["dielectric"], 0], np.float64)


# Scenes of at least this many triangles build their BVH on the GPU when one is usable (both builders give the same tree).
DEVICE_BVH_MIN_TRIS = 1 << 17


def default_bvh_builder(n_tris, device=0):
    """The builder flatten uses when it is given none: fspt_bvh_build_device on `device` for large scenes on a machine
    with a usable sm_100 device, the host builder otherwise.  A device build that fails raises; it is not retried on the
    host."""
    if n_tris >= DEVICE_BVH_MIN_TRIS and capi.device_usable(device):
        return functools.partial(capi.bvh_build_device, device=device)
    return capi.bvh_build


def flatten(triangle_sets, atlas, env, bins, normalize=None, n_threads=0, builder=None, device=0):
    """new BVH(geometry, 4) + serializeTree + the flatten loop (main.js:337-392) + light buffers (:394-401).
    builder: bvh_build-like callable; default default_bvh_builder(T, device)."""
    verts = np.concatenate([t.verts for t in triangle_sets], axis=0)
    build_verts = verts
    if normalize:
        # scene.normalize (main.js:337-348) rescales vertices AFTER Triangle.boundingBox was computed, so the
        # builder sees stale boxes; reproduced by building on the original verts and flattening the new ones.
        mn, mx = verts.reshape(-1, 3).min(axis=0), verts.reshape(-1, 3).max(axis=0)
        longest = float(max(max(mx[0] - mn[0], mx[1] - mn[1]), mx[2] - mn[2]))
        centroid = (mn + mx) * 0.5
        verts = (verts - centroid) * (2 * normalize / longest)
    builder = builder or default_bvh_builder(verts.shape[0], device)
    box = build_verts if normalize else None
    nodes, order, depth = (builder(verts, 4, n_threads, box_verts=box) if builder is capi.bvh_build
                           else builder(verts, 4, box_verts=box))
    normals = np.concatenate([t.normals for t in triangle_sets], axis=0)
    tangents = np.concatenate([t.tangents for t in triangle_sets], axis=0)
    bitangents = np.concatenate([t.bitangents for t in triangle_sets], axis=0)
    uvs = np.concatenate([t.uvs for t in triangle_sets], axis=0)
    mats = np.concatenate([np.repeat(material_row(t.material)[None, :], t.count, axis=0) for t in triangle_sets], axis=0)
    ntb = np.stack([normals, tangents, bitangents], axis=2)  # (T, vertex, {n,t,b}, 3): [n1 t1 b1 n2 t2 b2 ...]
    lights, ranges = [], []
    for t in triangle_sets:
        if sum(t.material["emittance"]) > 0:  # Vec3.dot(prop.emittance,[1,1,1]) > 0 (main.js:326)
            start = sum(l.shape[0] for l in lights)
            lights.append(t.verts.reshape(-1, 9))
            ranges += [start, start + t.count - 1]
    return SceneArrays(
        bvh=nodes,
        tris=verts[order].reshape(-1, 9).astype(np.float32),
        mats=mats[order].astype(np.float32),
        norms=ntb[order].reshape(-1, 27).astype(np.float32),
        uvs=uvs[order].reshape(-1, 6).astype(np.float32),
        atlas=atlas, env=env, bins=bins,
        lights=np.concatenate(lights, axis=0).astype(np.float32) if lights else None,
        light_ranges=np.asarray(ranges, np.float32) if ranges else None,
        depth=depth, order=order, verts64=verts[order].reshape(-1, 9))
