"""Scene-JSON front end: "drop a scene JSON in, get the same arrays main.js would upload" (SURVEY row f4).

Follows main.js (scene keys :67-73,289-348,869-871,929-948), obj_loader.js (OBJ text -> Triangle records),
mtl_loader.js (MTL tokens) and the asset handling of utility.js, with the browser replaced by the file system
and PIL.  Output = fspt_b200.scene.SceneArrays, i.e. exactly the buffers of SURVEY.md appendix A.
"""
import json
import math
import os

import numpy as np

from . import capi
from .geometry import mesh_to_triangles
from .scene import flatten, get_material
from .texture_packer import TexturePacker

SCALAR_TOKENS = {"ns", "ni", "d", "illum", "dielectric", "ior"}                       # mtl_loader.js:7
VECTOR_TOKENS = {"ka", "kd", "kem", "ks", "ke", "pr", "pm", "pmr", "pmr_swizzle"}      # mtl_loader.js:8
STRING_TOKENS = {"map_bump", "map_kd", "map_kem", "map_ks", "map_d", "map_ns", "map_pmr"}  # mtl_loader.js:9


def _js_parse_float(tok):
    """parseFloat: longest numeric prefix, NaN otherwise."""
    tok = tok.strip()
    best = float("nan")
    for n in range(len(tok), 0, -1):
        try:
            best = float(tok[:n])
            if tok[:n].lower() in ("inf", "+inf", "-inf", "nan", "infinity", "-infinity", "+infinity"):
                best = float("nan")
                continue
            break
        except ValueError:
            continue
    return best


def parse_materials(mtl_text, base_path):
    """ParseMaterials (mtl_loader.js:3-41) -> (materials dict, set of texture urls)."""
    materials, urls, name = {}, set(), None
    for line in mtl_text.split("\n"):
        tokens = [t for t in line.strip().split(" ") if t != ""] or [""]
        key = tokens[0].lower()
        if key == "newmtl":
            name = tokens[1]
            materials[name] = {}
        if name is None:
            continue
        value, is_url = None, False
        if key in SCALAR_TOKENS:
            value = _js_parse_float(tokens[1]) if len(tokens) > 1 else float("nan")
        elif key in VECTOR_TOKENS:
            value = [_js_parse_float(t) for t in tokens[1:]]
        elif key in STRING_TOKENS:
            value = tokens[1] if len(tokens) > 1 else None
            is_url = True
        if value is not None and value == value and value != 0 and value != "" and value != []:  # `if (value)`
            if is_url:
                urls.add(base_path + "/" + value)
            materials[name][key] = value
    return materials, urls


def parse_obj(obj_text, read_text, base_path, skips=()):
    """The line loop of parseMesh (obj_loader.js:164-192).  Returns vertices, uvs, mesh normals, faces (list of
    (group, [[v,vt,vn] x3]) after fan triangulation, obj_loader.js:54-60), group order, materials, urls."""
    vertices, uvs, mesh_normals, faces = [], [], [], []
    group, groups, materials, urls = "FSPT_DEFAULT_GROUP", [], {}, set()
    skips = set(skips or ())
    for line in obj_text.split("\n"):
        arr = [t for t in line.strip().split(" ") if t != ""]
        if not arr:
            continue
        vals = arr[1:]
        if arr[0] == "v":
            vertices.append([_js_parse_float(x) for x in vals[:3]])
        elif arr[0] == "f" and group not in skips:
            if group not in groups:
                groups.append(group)
            idx = [[_js_parse_float(x) for x in s.split("/")] for s in vals]
            # relative (negative / zero) indices resolve against the vertices and normals read SO FAR
            # (parseTriangle, obj_loader.js:107-113: `vertices.length + idx + 1` at the time of the face line)
            for c in idx:
                if c[0] < 1:
                    c[0] = len(vertices) + c[0] + 1
                if len(c) > 2 and c[2] == c[2] and c[2] < 1:
                    c[2] = len(mesh_normals) + c[2] + 1
            for i in range(len(idx) - 2):  # parseFace
                faces.append((group, [list(idx[0]), list(idx[i + 1]), list(idx[i + 2])]))
        elif arr[0] == "vt":
            uv = [(_js_parse_float(x) if _js_parse_float(x) == _js_parse_float(x) and _js_parse_float(x) != 0 else 0.0) for x in vals]
            uvs.append(uv[:2])
        elif arr[0] == "vn":
            mesh_normals.append([_js_parse_float(x) for x in vals])
        elif arr[0] == "usemtl":
            group = " ".join(arr[1:])
        elif arr[0] == "mtllib":
            materials, urls = parse_materials(read_text(base_path + "/" + " ".join(arr[1:])), base_path)
    return dict(vertices=np.asarray(vertices, np.float64).reshape(-1, 3), uvs=uvs, mesh_normals=mesh_normals,
                faces=faces, groups=groups, materials=materials, urls=urls)


def obj_to_triangle_sets(parsed, prop, world_transforms):
    """parseTriangle + smooth normals + calcTangents for every group of one OBJ (obj_loader.js:103-212).
    Smooth normals are averaged over ALL faces of the OBJ that share a vertex index, in file order."""
    V = parsed["vertices"]
    vi, ti, ni, gid = [], [], [], []
    gindex = {g: k for k, g in enumerate(parsed["groups"])}
    for g, tri in parsed["faces"]:
        row_v, row_t, row_n = [], [], []
        for c in tri:
            row_v.append(int(c[0]) - 1)                 # relative indices were resolved while parsing the face line
            t = c[1] if len(c) > 1 else float("nan")
            row_t.append(int(t) - 1 if t == t else -1)  # vt indices are used as given (obj_loader.js:109-110)
            n = c[2] if len(c) > 2 else float("nan")
            row_n.append(int(n) - 1 if n == n else -1)
        vi.append(row_v); ti.append(row_t); ni.append(row_n); gid.append(gindex[g])
    vi, ti, ni, gid = np.asarray(vi, np.int64), np.asarray(ti, np.int64), np.asarray(ni, np.int64), np.asarray(gid)
    has_uv = len(parsed["uvs"]) > 0 and np.all(ti >= 0)
    face_uvs = np.asarray(parsed["uvs"], np.float64)[ti] if has_uv else None
    ts = mesh_to_triangles(V, vi, prop, world_transforms, face_uvs,
                           np.asarray(parsed["mesh_normals"], np.float64) if parsed["mesh_normals"] else None, ni)
    out = []
    from .geometry import TriangleSet
    for k, g in enumerate(parsed["groups"]):
        m = gid == k
        out.append((g, TriangleSet(ts.verts[m], ts.normals[m], ts.tangents[m], ts.bitangents[m], ts.uvs[m])))
    return out


def load_image(path):
    """Image element -> RGBA8 (h,w,4), row 0 = top."""
    from PIL import Image
    img = Image.open(path).convert("RGBA")
    return {"src": path, "pixels": np.asarray(img, np.uint8).copy()}


def canvas_roundtrip(rgba):
    """ctx.drawImage + getImageData (env_sampler.js:55-60): canvases store premultiplied 8-bit pixels, so the
    RGB of an RGBE texel is quantised by its 'alpha' (the exponent byte) before ProcessEnvRadiance sees it."""
    a = rgba[..., 3:4].astype(np.float64)
    pre = np.floor(rgba[..., :3].astype(np.float64) * a / 255.0 + 0.5)
    with np.errstate(divide="ignore", invalid="ignore"):
        un = np.where(a > 0, np.floor(pre * 255.0 / a + 0.5), 0.0)
    out = rgba.copy()
    out[..., :3] = np.clip(un, 0, 255).astype(np.uint8)
    return out


def compile_scene(scene, asset_root, read_text=None, load_img=None, n_threads=0, emulate_canvas=True, device=0):
    """initBVH (main.js:284-445).  scene: dict (parsed JSON).  Returns (SceneArrays, camera dict).
    device: the CUDA device a large scene's BVH may be built on (scene.default_bvh_builder)."""
    read_text = read_text or (lambda p: open(os.path.join(asset_root, p)).read())
    load_img = load_img or (lambda p: load_image(os.path.join(asset_root, p)))
    env = scene.get("environment")
    if isinstance(env, str):
        e = load_img(env)["pixels"]
        bins = capi.env_bins(canvas_roundtrip(e) if emulate_canvas else e)
        env_px = e
    elif isinstance(env, list):
        # createEnvironmentMapPixels (main.js:182-204): an RGB32F gradient whose alpha reads 1.0, so envColor's
        # 2^(a*255-128) saturates every non-zero stop to the 1024 clamp -- only black is meaningful
        if any(abs(float(c)) > 0 for stop in env for c in stop):
            raise NotImplementedError("colour-stop environments saturate in the reference (SURVEY A.2); use an RGBE image")
        env_px = np.zeros((2048, 1, 4), np.uint8)
        bins = np.array([[0, 0, 1, 2048]], np.uint16)
    else:
        raise ValueError("scene.environment is mandatory: without it the reference's tracer.fs does not compile (main.js:303-308)")
    props = list(scene.get("props") or []) + list(scene.get("static_props") or []) + \
        list((scene.get("animated_props") or {}).values() if isinstance(scene.get("animated_props"), dict)
             else (scene.get("animated_props") or []))                                   # mergeSceneProps, main.js:869-871
    packer = TexturePacker(scene.get("atlasRes") or 2048)                                  # main.js:39,948
    assets, sets = {}, []

    def asset(url):
        if url not in assets:
            assets[url] = load_img(url)
        return assets[url]
    for prop in props:
        for k in ("diffuse", "metallicRoughness", "normal", "emission"):
            if isinstance(prop.get(k), str):
                asset(prop[k])
        base = "/".join(prop["path"].split("/")[:-1])
        p = dict(prop)
        p.setdefault("rotate", [])
        parsed = parse_obj(read_text(prop["path"]), read_text, base, prop.get("skips"))
        for url in sorted(parsed["urls"]):
            asset(url)
        for gname, ts in obj_to_triangle_sets(parsed, p, scene.get("worldTransforms")):
            ts.material = get_material(p, parsed["materials"].get(gname, {}), packer, assets, base)
            sets.append(ts)
    packer.setAndGetResolution()
    sa = flatten(sets, packer.getPixels(), env_px, bins, normalize=scene.get("normalize"), n_threads=n_threads,
                 device=device)
    cam = dict(eye=scene.get("cameraPos") or [0, 0, 2], dir=scene.get("cameraDir") or [0, 0, -1],
               fov_scale=scene.get("fovScale") or 0.5, env_theta=scene.get("environmentTheta") or 0,
               aperture=0.02, focal_depth=2.0, exposure=scene.get("exposure") or 1.0,
               samples=scene.get("samples") or 2000)                                     # main.js:67-74, index.html:25,27
    return sa, cam


def load_scene(scene_path, asset_root=None, **kw):
    asset_root = asset_root or os.path.dirname(os.path.dirname(os.path.abspath(scene_path)))
    with open(scene_path) as f:
        return compile_scene(json.load(f), asset_root, **kw)


def autofocus_distance(verts, eye, direction, max_t=1e6):
    """shootAutoFocusRay (main.js:447-546) in float64 with the reference's epsilon 1e-12.  The JS walks its tree;
    pruning is conservative, so the closest distance equals this vectorised pass over all triangles."""
    v = np.asarray(verts, np.float64).reshape(-1, 3, 3)
    eye, d = np.asarray(eye, np.float64), np.asarray(direction, np.float64)
    eps = 1e-12
    e1, e2 = v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]
    p = np.stack([d[1] * e2[:, 2] - d[2] * e2[:, 1], -(d[0] * e2[:, 2] - d[2] * e2[:, 0]), d[0] * e2[:, 1] - d[1] * e2[:, 0]], 1)
    det = (e1 * p).sum(1)
    ok = ~((det > -eps) & (det < eps))
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = 1.0 / det
        t = eye - v[:, 0]
        u = (t * p).sum(1) * inv
        ok &= ~((u < 0) | (u > 1))
        q = np.stack([t[:, 1] * e1[:, 2] - t[:, 2] * e1[:, 1], -(t[:, 0] * e1[:, 2] - t[:, 2] * e1[:, 0]), t[:, 0] * e1[:, 1] - t[:, 1] * e1[:, 0]], 1)
        w = (q * d).sum(1) * inv
        ok &= ~((w < 0) | (u + w > 1))
        dist = (e2 * q).sum(1) * inv
        ok &= dist > eps
    return float(dist[ok].min()) if ok.any() else float(max_t)
