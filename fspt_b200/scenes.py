"""The benchmark / parity scenes of BASELINE.json, built from procedural assets (the reference ships neither
bunny_big.obj nor its HDRi, see .MISSING_LARGE_BLOBS), through the same compile path a scene JSON takes."""
import numpy as np

from . import capi, procedural as pr
from .geometry import mesh_to_triangles
from .scene import flatten, get_material
from .texture_packer import TexturePacker

# camera / env of scene/bunny.json:3-5 and the DOM defaults (index.html:25,27; main.js:69-74)
BUNNY_CAMERA = dict(eye=[-0.751, 0.665, 1.820], dir=[0.304, -0.489, -0.818], fov_scale=0.5, env_theta=1.66,
                    aperture=0.02, focal_depth=2.0)


def _env(env_size, kind="sun", host=None):
    w, h = env_size
    env = pr.environment(w, h) if kind == "sun" else pr.constant_environment(w, h, kind)
    return env, (host or capi).env_bins(env)


def bunny_class(subdiv=6, atlas_res=2048, env_size=(2048, 1024), textured=True, host=None, device=0):
    """scene/bunny.json with the missing bunny replaced by a lumpy icosphere (20*4^subdiv triangles) and the
    dungeon maps by procedural PBR maps.  Props, transforms and material constants follow scene/bunny.json:6-41.
    host: the module that supplies the host-side scene compilers bvh_build / env_bins / pack_layer -- default the
    product's native ones (capi); the reference arm of bench.py passes the oracle so that it never loads the product."""
    v, f = pr.icosphere(subdiv)
    props = [
        dict(mesh=(pr.lumpy(v), f, None), scale=0.35, rotate=[{"angle": 0, "axis": [0, 0, 1]}], translate=[0.1, -0.4, 0],
             diffuse=[1, 1, 1], emittance=[0, 0, 0], metallicRoughness=[0, 0.1, 0], ior=1.4, normals="smooth"),
        dict(mesh=(pr.QUAD_VERTS, pr.QUAD_FACES, pr.QUAD_FACE_UVS), scale=4, rotate=[{"angle": 3.1415, "axis": [0, 0, 1]}],
             translate=[0, -0.75, 0], emittance=[0, 0, 0], normals="flat",
             diffuse="A/baseColor", metallicRoughness="A/metallicRoughness", normal="A/normal"),
        dict(mesh=(pr.QUAD_VERTS, pr.QUAD_FACES, pr.QUAD_FACE_UVS), scale=4, rotate=[{"angle": -1.57, "axis": [1, 0, 0]}],
             translate=[0, 0.25, -1], emittance=[0, 0, 0], normals="flat", ior="10",
             emission="B/emissive", diffuse="B/baseColor", metallicRoughness="B/metallicRoughness", normal="B/normal"),
    ]
    assets = {}
    if textured:
        for tag, seed in (("A", 7), ("B", 11)):
            for k, img in pr.pbr_maps(atlas_res, seed, tag).items():
                assets["%s/%s" % (tag, k)] = img
    else:
        for p in props[1:]:
            for k in ("diffuse", "metallicRoughness", "normal", "emission"):
                p.pop(k, None)
    return compile_props(props, assets, atlas_res, _env(env_size, host=host), host=host, device=device), dict(BUNNY_CAMERA)


def compile_props(props, assets, atlas_res, env_and_bins, n_threads=0, builder=None, host=None, device=0):
    packer = TexturePacker(atlas_res, pack_layer=host.pack_layer if host else None)
    if host is not None and builder is None:
        builder = host.bvh_build
    sets = []
    for p in props:
        vtx, faces, face_uvs = p["mesh"]
        ts = mesh_to_triangles(vtx, faces, p, None, face_uvs)
        ts.material = get_material(p, {}, packer, assets)
        sets.append(ts)
    packer.setAndGetResolution()
    atlas = packer.getPixels()
    env, bins = env_and_bins
    return flatten(sets, atlas, env, bins, n_threads=n_threads, builder=builder, device=device)


def quad_scene(env_size=(64, 32)):
    """asset_packs/misc/top_mono.obj alone (2 triangles => the root is a leaf): the hand-checkable KAT."""
    p = dict(mesh=(pr.QUAD_VERTS, pr.QUAD_FACES, pr.QUAD_FACE_UVS), scale=1, rotate=[], translate=[0, 0, 0],
             emittance=[0, 0, 0], normals="flat", diffuse=[0.8, 0.8, 0.8])
    return compile_props([p], {}, 4, _env(env_size)), dict(eye=[0, 2, 0], dir=[0, -1, 0.0001], fov_scale=0.5,
                                                           env_theta=0.0, aperture=0.0, focal_depth=2.0)


def sphere_soup_verts(subdiv=7, n_soup=672320, seed=1234):
    """The (T, 9) float64 vertices sphere_soup builds its BVH from (the inputs of BVH builder measurements and tests)."""
    props = _sphere_soup_props(subdiv, n_soup, seed, 0.8)
    return np.concatenate([mesh_to_triangles(p["mesh"][0], p["mesh"][1], p).verts for p in props], axis=0)


def _sphere_soup_props(subdiv, n_soup, seed, albedo):
    v, f = pr.icosphere(subdiv)
    props = [dict(mesh=(v, f, None), scale=0.5, rotate=[], translate=[0, 0, 0], diffuse=[albedo] * 3,
                  emittance=[0, 0, 0], metallicRoughness=[0, 1.0, 0], normals="smooth")]
    sa_props = props
    if n_soup:
        soup = pr.triangle_soup(n_soup, seed)
        sv = soup.reshape(-1, 3)
        sf = np.arange(sv.shape[0], dtype=np.int64).reshape(-1, 3)
        sa_props = props + [dict(mesh=(sv, sf, None), scale=1, rotate=[], translate=[0, 0, 0], diffuse=[albedo] * 3,
                                 emittance=[0, 0, 0], metallicRoughness=[0, 1.0, 0], normals="flat")]
    return sa_props


def sphere_soup(subdiv=7, n_soup=672320, seed=1234, env_size=(2048, 1024), albedo=0.8, device=0):
    """BASELINE config 3: subdivided icosphere + uniform random triangle soup, Lambert rho = 0.8, aperture 0."""
    sa_props = _sphere_soup_props(subdiv, n_soup, seed, albedo)
    cam = dict(eye=[0, 0.3, 2.6], dir=[0, -0.1, -1], fov_scale=0.5, env_theta=0.25, aperture=0.0, focal_depth=2.0)
    return compile_props(sa_props, {}, 4, _env(env_size), device=device), cam


def pbr_scene(atlas_res=2048, subdiv=5, env_size=(2048, 1024), device=0):
    """BASELINE config 4: textured quads + spheres with all four maps + one refractive prop (dielectric >= 0)."""
    v, f = pr.icosphere(subdiv)
    assets = {}
    for tag, seed in (("A", 7), ("B", 11)):
        for k, img in pr.pbr_maps(atlas_res, seed, tag).items():
            assets["%s/%s" % (tag, k)] = img
    props = [
        dict(mesh=(pr.QUAD_VERTS, pr.QUAD_FACES, pr.QUAD_FACE_UVS), scale=6, rotate=[{"angle": 3.1415, "axis": [0, 0, 1]}],
             translate=[0, -0.75, 0], emittance=[0, 0, 0], normals="flat", diffuse="A/baseColor",
             metallicRoughness="A/metallicRoughness", normal="A/normal"),
        dict(mesh=(pr.QUAD_VERTS, pr.QUAD_FACES, pr.QUAD_FACE_UVS), scale=6, rotate=[{"angle": -1.57, "axis": [1, 0, 0]}],
             translate=[0, 0.25, -1.5], emittance=[0, 0, 0], normals="flat", emission="B/emissive", diffuse="B/baseColor",
             metallicRoughness="B/metallicRoughness", normal="B/normal"),
        dict(mesh=(v, f, None), scale=0.4, rotate=[], translate=[-0.6, -0.35, 0.2], emittance=[0, 0, 0], normals="smooth",
             diffuse="B/baseColor", metallicRoughness="B/metallicRoughness", normal="B/normal"),
        dict(mesh=(v, f, None), scale=0.35, rotate=[], translate=[0.45, -0.4, 0.4], emittance=[0, 0, 0], normals="smooth",
             diffuse=[0.9, 0.95, 1.0], metallicRoughness=[0, 0.05, 0], ior=1.4, dielectric=0.5),
        dict(mesh=(pr.lumpy(v), f, None), scale=0.3, rotate=[], translate=[0.0, -0.45, -0.5], emittance=[0, 0, 0],
             normals="smooth", diffuse=[1.0, 0.8, 0.3], metallicRoughness=[1.0, 0.25, 0]),
    ]
    cam = dict(eye=[-0.2, 0.35, 2.0], dir=[0.08, -0.3, -1.0], fov_scale=0.5, env_theta=1.66, aperture=0.01, focal_depth=2.0)
    return compile_props(props, assets, atlas_res, _env(env_size), device=device), cam


def lens_features(cam):
    """[1 - 1/focalDepth, aperture] (main.js:74)."""
    return [1.0 - 1.0 / float(cam["focal_depth"]), float(cam["aperture"])]


def rand_bases(n, seed):
    """`Math.random()*10000` streams for drawCamera and drawTracer (main.js:748,777), seeded (mulberry32)."""
    def mulberry32(a):
        while True:
            a = (a + 0x6D2B79F5) & 0xFFFFFFFF
            t = a
            t = ((t ^ (t >> 15)) * (t | 1)) & 0xFFFFFFFF
            t ^= (t + (((t ^ (t >> 7)) * (t | 61)) & 0xFFFFFFFF)) & 0xFFFFFFFF
            yield ((t ^ (t >> 14)) & 0xFFFFFFFF) / 4294967296.0
    g = mulberry32(seed & 0xFFFFFFFF)
    cam, tr = [], []
    for _ in range(n):       # tick(): drawCamera() then drawTracer(), one Math.random() each
        cam.append(next(g) * 10000.0)
        tr.append(next(g) * 10000.0)
    return np.asarray(cam, np.float32), np.asarray(tr, np.float32)
