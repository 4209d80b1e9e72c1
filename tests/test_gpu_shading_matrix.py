"""The shading kernel on crafted scenes: the material, texture-layer, UV, normal and environment edges of tracer.fs's
loop body (csrc/shade.cuh shade_hit) that the procedural BASELINE scenes reach rarely or never.

Every case is a small hand-made scene (64x48 pixels, 3 ticks) compiled through scene.flatten with a hand-made atlas of
R x R layers, R = 32 (REPEAT wraps with a mask) and R = 24 (REPEAT wraps with a modulo):
  * materials     metallic {0, 0.5, 1} x roughness {0, 1/255, 0.5, 1} (roughness 0 and 1/255 sit under the 0.001 floor);
  * dielectrics   spheres with dielectric {0, 0.5, 3} x ior {1.0, 0.7, 1.4, 2.4}: ior 1 (Schlick's 0 / 2), ior < 1
                  (total internal reflection from outside), refraction caps 0, 1 and 64;
  * inside_sphere the camera inside a closed non-dielectric sphere: Beer's law with a negative dielectric grows the
                  throughput above 1;
  * back_quads    open quads seen from the back;
  * emission      emissive layer 255 on diffuse 255;
  * normals       normal-map texels that tilt the macro normal hard or lay it in the tangent plane, geometric normals
                  (0,0,+-1) and normals with z = 0.999f and its neighbours (the switch of the tangent frame);
  * layers        one textured map per role in each role in turn, one layer in two roles, two triangle sets with the
                  same layer quadruple, and layers that differ from texel 0 in one texel only (the first, the last, the
                  first of a band of the host's constant-layer scan, and one that differs in alpha only);
  * uvs           UV offsets -0.5, -3.25 and 17, UV scales up to 1e6 and one triangle whose uv * R exceeds 1e9;
  * env_top, env_bottom, env_const   environments whose only bright texels lie in the top or the bottom row
                  (sinPhi -> 0 in envPdf), and a constant one.

The checks, all bit for bit:
  * the CUDA path against the oracle: RGBA accumulator, last sample colour, ray / node / leaf counts and capped paths,
    on both atlas forms (material-interleaved and plain), with NaN sanitising on and off and any-hit on and off;
  * the oracle against what the reference's own tracer.fs computed on the same cases
    (tests/golden/reference_shaders/shading_matrix.npz, generator tests/golden/make_shading_matrix.py), and the CUDA
    path against those records;
  * each case reaches its branch: changing the feature changes the oracle image, and no per-sample colour comes near the
    1024 clamp of the accumulation, so the clamp hides nothing.
"""
import dataclasses
import functools
import os
import sys

import numpy as np
import pytest

from fspt_b200 import capi, scenes, procedural as pr
from fspt_b200.geometry import TriangleSet, mesh_to_triangles
from fspt_b200.scene import flatten

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_reference_outputs as golden  # noqa: E402

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_shaders", "shading_matrix.npz")
W, H, TICKS, SEED = 64, 48, 3, 57
R_SIZES = (32, 24)
UNCAPPED = 1 << 20  # the oracle's refraction cap that no path of these scenes reaches (the reference has none)
CUDA_UNCAPPED = 30000  # the API's maximum
CAM = dict(eye=[0.0, 0.0, 3.0], dir=[0.0, 0.0, -1.0], fov_scale=0.5, env_theta=0.3, aperture=0.0, focal_depth=2.0)


# ---------------------------------------------------------------------------------------------------------------------
# scene pieces
class Atlas:
    """Hand-made R x R RGBA8 layers; add() returns the layer index a material refers to."""

    def __init__(self, R):
        self.R, self.layers = R, []

    def add(self, img):
        self.layers.append(np.ascontiguousarray(img, np.uint8))
        return len(self.layers) - 1

    def const(self, rgb, alpha=255):
        img = np.empty((self.R, self.R, 4), np.uint8)
        img[...] = list(rgb) + [alpha]
        return self.add(img)

    def noise(self, seed):
        img = np.random.default_rng(seed).integers(0, 256, (self.R, self.R, 4), dtype=np.uint8)
        img[..., 3] = 255
        return self.add(img)

    def one_texel(self, i, rgba, base=(90, 90, 90, 255)):
        """A layer equal to `base` everywhere but flat texel i (row-major, row = GL row)."""
        img = np.empty((self.R, self.R, 4), np.uint8)
        img[...] = base
        img.reshape(-1, 4)[i] = rgba
        return self.add(img)

    def array(self):
        return np.stack(self.layers)


def material(diffuse, emission, mr, normal, ior=1.4, dielectric=-1.0):
    return {"diffuseIndex": diffuse, "specularIndex": emission, "roughnessIndex": mr, "normalIndex": normal,
            "ior": float(ior), "dielectric": float(dielectric), "emittance": [0.0, 0.0, 0.0]}


def quad_at(P, mat, uv=(0.0, 0.0, 1.0, 1.0), n=(0, 0, 1), t=(1, 0, 0), b=(0, 1, 0)):
    """Two triangles over the corners P[0..3] (UV corners (u0, v0), (u1, v0), (u1, v1), (u0, v1)), one normal, tangent
    and bitangent for every vertex."""
    u0, v0, u1, v1 = uv
    UV = np.array([[u0, v0], [u1, v0], [u1, v1], [u0, v1]], np.float64)
    f = np.array([[0, 1, 2], [0, 2, 3]])
    frame = [np.broadcast_to(np.asarray(a, np.float64), (2, 3, 3)).copy() for a in (n, t, b)]
    return TriangleSet(np.asarray(P, np.float64)[f], frame[0], frame[1], frame[2], UV[f], material=mat)


def quad(x0, y0, x1, y1, z, mat, **kw):
    """A quad in the plane z, counter-clockwise seen from +z (the camera's side)."""
    return quad_at([[x0, y0, z], [x1, y0, z], [x1, y1, z], [x0, y1, z]], mat, **kw)


def floor_quad(mat, y=-1.2):
    return quad_at([[-3, y, 2], [3, y, 2], [3, y, -4], [-3, y, -4]], mat, uv=(0, 0, 2, 2), n=(0, 1, 0), b=(0, 0, -1))


def sphere(center, radius, mat, subdiv=2):
    v, f = pr.icosphere(subdiv)
    ts = mesh_to_triangles(v, f, dict(scale=radius, translate=list(center), rotate=[], normals="smooth"))
    ts.material = mat
    return ts


def grid(cols, rows, i, size=0.9, span=(4.0, 3.0)):
    """Cell i of a cols x rows grid over the visible part of the plane z = 0: (x0, y0, x1, y1)."""
    cw, ch = span[0] / cols, span[1] / rows
    cx, cy = -span[0] / 2 + cw * (i % cols + 0.5), span[1] / 2 - ch * (i // cols + 0.5)
    return cx - cw * size / 2, cy - ch * size / 2, cx + cw * size / 2, cy + ch * size / 2


def _env(kind="sun"):
    w, h = 64, 32
    if kind == "sun":
        env = pr.environment(w, h, sun=(0.3, 0.3), sun_radius=0.06, sun_radiance=30.0)
    elif kind == "const":
        env = pr.constant_environment(w, h, 0.7)
    else:  # the only bright texels in the top or the bottom row
        rgb = np.full((h, w, 3), 0.05)
        rgb[0 if kind == "top" else h - 1] = (40.0, 30.0, 20.0)
        env = pr._rgbe_encode(rgb)
    return env, capi.env_bins(env)


class Base:
    """The layers most materials share."""

    def __init__(self, A):
        self.grey = A.const((200, 200, 200))
        self.black = A.const((0, 0, 0))
        self.mr = A.const((0, 128, 0))
        self.flat = A.const((128, 128, 255))
        self.noise = A.noise(5)

    def mat(self, diffuse=None, emission=None, mr=None, normal=None, **kw):
        return material(self.grey if diffuse is None else diffuse, self.black if emission is None else emission,
                        self.mr if mr is None else mr, self.flat if normal is None else normal, **kw)


# ---------------------------------------------------------------------------------------------------------------------
# the cases: (triangle sets, atlas, environment kind, info); info names the pieces the reach checks change
def case_materials(A, B):
    sets, info = [], {}
    for row, metal in enumerate((0, 128, 255)):
        for col, rough in enumerate((0, 1, 128, 255)):
            layer = A.const((metal, rough, 0))
            info["mr/%d/%d" % (metal, rough)] = layer
            sets.append(quad(*grid(4, 3, 4 * row + col), 0.0, B.mat(diffuse=B.noise, mr=layer)))
    sets.append(floor_quad(B.mat()))
    return sets, "sun", info


DIELECTRICS = (0.0, 0.5, 3.0)
IORS = (1.0, 0.7, 1.4, 2.4)


def case_dielectrics(A, B):
    sets = []
    smooth = A.const((0, 13, 0))
    for row, diel in enumerate(DIELECTRICS):
        for col, ior in enumerate(IORS):
            x0, y0, x1, y1 = grid(4, 3, 4 * row + col)
            sets.append(sphere(((x0 + x1) / 2, (y0 + y1) / 2, 0.0), 0.42,
                               B.mat(diffuse=A.const((230, 200, 160)), mr=smooth, ior=ior, dielectric=diel)))
    sets.append(quad(-4, -3, 4, 3, -1.5, B.mat(diffuse=B.noise), uv=(0, 0, 3, 2)))
    return sets, "sun", {}


def case_inside_sphere(A, B):
    """The camera inside a closed sphere of a non-dielectric material: every hit is an inside hit, Beer's law with
    dielectric -1 multiplies the throughput by 1 + (1 - diffuse) * t > 1, the glow comes from a faint emission layer."""
    m = B.mat(diffuse=A.const((200, 170, 230)), emission=A.const((6, 5, 4)), mr=A.const((40, 160, 0)))
    return [sphere((0.0, 0.0, 2.6), 1.3, m, subdiv=3)], "sun", {}


def case_back_quads(A, B):
    """Open quads whose stored normal faces away from the camera (inside hits), non-dielectric and dielectric."""
    sets = []
    for i, (diel, ior) in enumerate(((-1.0, 1.4), (-0.25, 2.4), (0.0, 1.4), (2.0, 0.7))):
        sets.append(quad(*grid(2, 2, i), 0.0, B.mat(diffuse=B.noise, ior=ior, dielectric=diel), n=(0, 0, -1)))
    sets.append(floor_quad(B.mat()))
    return sets, "sun", {}


def case_emission(A, B):
    info = {"emission": A.const((255, 255, 255))}
    white = A.const((255, 255, 255))
    sets = [quad(-1.8, -1.0, -0.2, 1.0, 0.0, B.mat(diffuse=white, emission=info["emission"])),
            quad(0.2, -1.0, 1.8, 1.0, -0.5, B.mat(diffuse=B.noise)),
            floor_quad(B.mat(diffuse=white))]
    return sets, "sun", info


NORMAL_TEXELS = ((128, 128, 255), (255, 128, 128), (128, 128, 0), (0, 0, 128))


def case_normals(A, B):
    sets, info = [], {}
    for i, texel in enumerate(NORMAL_TEXELS):
        info["normal/%d" % i] = A.const(texel)
        sets.append(quad(*grid(4, 2, i), 0.0, B.mat(diffuse=B.noise, mr=A.const((0, 90, 0)), normal=info["normal/%d" % i])))
    z0 = np.float32(0.999)
    for i, z in enumerate((np.nextafter(z0, np.float32(0)), z0, np.nextafter(z0, np.float32(1)))):
        # zero tangent and bitangent: the macro normal is the interpolated geometric normal, renormalised, so |n.z| lands
        # within rounding of the tangent frame's 0.999f switch
        n = (float(np.sqrt(np.float64(1) - np.float64(z) ** 2)), 0.0, float(z))
        sets.append(quad(*grid(4, 2, 4 + i), 0.0, B.mat(diffuse=B.noise, mr=A.const((0, 90, 0))), n=n, t=(0, 0, 0), b=(0, 0, 0)))
    sets.append(quad(*grid(4, 2, 7), 0.0, B.mat(diffuse=B.noise), n=(0, 0, -1)))  # geometric (0, 0, -1)
    return sets, "sun", info


def scan_texels(R):
    """Flat texel indices the constant-layer scan must see: the first, the last, and the first of scan band 3
    (layer_texels * b / 8 in fspt_api.cu scan_layer_band)."""
    return {"first": 0, "last": R * R - 1, "band": R * R * 3 // 8}


def _uv_box(i, R):
    """UV rectangle around the centre of flat texel i (a sub-texel footprint: the texel dominates every tap)."""
    x, y = i % R, i // R
    return ((x + 0.3) / R, (y + 0.3) / R, (x + 0.7) / R, (y + 0.7) / R)


def case_layers(A, B):
    R = A.R
    sets, info = [], {}
    tex = [A.noise(11), A.noise(12), A.noise(13), A.noise(14)]
    for role in range(4):  # diffuse, emission, metallic-roughness, normal: one textured map, three colour layers
        args = [None] * 4
        args[role] = tex[role]
        if role == 1:  # a dim emission layer keeps the sample colours far from the clamp
            args[role] = A.add(np.minimum(A.layers[tex[1]], 40))
        sets.append(quad(*grid(4, 3, role), 0.0, B.mat(*args)))
    sets.append(quad(*grid(4, 3, 4), 0.0, B.mat(diffuse=tex[3], normal=tex[3])))  # one layer in two roles
    same = B.mat(diffuse=tex[0], mr=tex[2])
    sets.append(quad(*grid(4, 3, 5), 0.0, same))                                   # two triangle sets, one quadruple
    sets.append(quad(*grid(4, 3, 6), 0.0, dict(same), uv=(0.3, 0.1, 0.8, 0.9)))
    cell = 7
    for name, i in scan_texels(R).items():
        info["scan/" + name] = layer = A.one_texel(i, (250, 30, 140, 255))
        sets.append(quad(*grid(4, 3, cell), 0.0, B.mat(diffuse=layer), uv=_uv_box(i, R)))
        cell += 1
    info["scan/alpha"] = layer = A.one_texel(R * R // 2 + 5, (90, 90, 90, 17))
    sets.append(quad(*grid(4, 3, cell), 0.0, B.mat(diffuse=layer), uv=_uv_box(R * R // 2 + 5, R)))
    return sets, "sun", info


UV_RECTS = ((-0.5, -0.5, 0.5, 0.5), (-3.25, -3.25, -2.25, -2.25), (17.0, 17.0, 18.0, 18.0), (0.0, 0.0, 1e3, 1e3),
            (0.0, 0.0, 1e6, 1e6), (-1e6, -1e6, 0.0, 1e6))


def case_uvs(A, B):
    sets = [quad(*grid(4, 2, i), 0.0, B.mat(diffuse=B.noise, normal=A.noise(21)), uv=uv) for i, uv in enumerate(UV_RECTS)]
    # one triangle with uv * R above 1e9 (the +-1e9 guard of coord_to_i32)
    x0, y0, x1, y1 = grid(4, 2, 6, size=1.8)
    huge = quad(x0, y0, x1, y1, 0.0, B.mat(diffuse=B.noise), uv=(1e8, 2e8, 1e8 + 64.0, 2e8 + 64.0))
    for name in ("verts", "normals", "tangents", "bitangents", "uvs"):
        setattr(huge, name, getattr(huge, name)[:1].copy())
    sets.append(huge)
    return sets, "sun", {}


def _env_case(kind):
    def build(A, B):
        metal = A.const((255, 20, 0))
        sets = [quad(-1.9, -1.0, -0.1, 1.0, 0.0, B.mat(diffuse=B.noise)),
                sphere((0.9, 0.0, 0.0), 0.8, B.mat(diffuse=A.const((220, 220, 220)), mr=metal), subdiv=3),
                floor_quad(B.mat())]
        return sets, kind, {}
    return build


CASES = {
    "materials": case_materials, "dielectrics": case_dielectrics, "inside_sphere": case_inside_sphere,
    "back_quads": case_back_quads, "emission": case_emission, "normals": case_normals, "layers": case_layers,
    "uvs": case_uvs, "env_top": _env_case("top"), "env_bottom": _env_case("bottom"), "env_const": _env_case("const"),
}
CAPS = {"dielectrics": (0, 1, 64)}  # refraction caps the CUDA path is held to the oracle at (default: 64)
IDS = [(name, R) for name in CASES for R in R_SIZES]


@functools.lru_cache(maxsize=None)
def build_case(name, R):
    """(SceneArrays, camera, info) of case `name` with an R x R atlas."""
    A = Atlas(R)
    B = Base(A)
    sets, env_kind, info = CASES[name](A, B)
    env, bins = _env(env_kind)
    sa = flatten(sets, A.array(), env, bins, builder=capi.bvh_build)
    return sa, dict(CAM), info


def primary(oracle_mod, cam, rb):
    return oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rb)


def oracle_run(oracle_mod, sa, cam, sanitize=0, max_refractions=UNCAPPED, ticks=TICKS):
    """The oracle over `ticks` ticks: (accumulator after each tick, last per-sample colour, summed counters)."""
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(ticks, SEED)
    fbs, col, tot = [], None, dict(rays=0, node_visits=0, leaf_visits=0, capped=0)
    for k in range(ticks):
        pos, d = primary(oracle_mod, cam, rc[k])
        fb, col, st = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fbs[-1] if fbs else None,
                              sanitize=sanitize, max_refractions=max_refractions, want_color=True)
        fbs.append(fb)
        for key in tot:
            tot[key] += st[key]
    return fbs, col, tot


@functools.lru_cache(maxsize=None)
def oracle_case(name, R, sanitize=0, max_refractions=UNCAPPED):
    import oracle
    sa, cam, _ = build_case(name, R)
    return oracle_run(oracle, sa, cam, sanitize, max_refractions)


def record_key(name, R, tick):
    return "shading/%s/R%d/tick%d" % (name, R, tick)


def record_keys():
    return [record_key(name, R, k) for name, R in IDS for k in range(TICKS)]


def bits_equal(a, b):
    return golden.beq(np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32))


def assert_bit_equal(got, ref, what):
    got, ref = np.ascontiguousarray(got, np.float32), np.ascontiguousarray(ref, np.float32)
    same = golden.canonical(got) == golden.canonical(ref)
    if not same.all():
        i = tuple(np.argwhere(~same)[0])
        raise AssertionError("%s: %d of %d differ; first at %s: got %r, oracle %r" % (what, int((~same).sum()), same.size,
                                                                                      i, got[i], ref[i]))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the cases are what they claim to be
@pytest.mark.parametrize("name,R", IDS)
def test_oracle_against_the_reference_shaders(name, R):
    """The oracle (no NaN sanitising, no effective refraction cap) against the stored output of tracer.fs itself."""
    fbs, _, _ = oracle_case(name, R)
    for k, fb in enumerate(fbs):
        golden.check(record_key(name, R, k), fb, path=PATH)


@pytest.mark.parametrize("name,R", IDS)
def test_sample_colours_stay_below_the_clamp(name, R):
    """tracer.fs:515 clamps each sample to [0, 1024] before it is accumulated: a wrong firefly above the clamp would
    look like a right one.  No sample of these cases comes near it, and the image is not black."""
    _, col, _ = oracle_case(name, R)
    rgb = col[..., :3]
    assert np.nanmax(rgb) < 256.0, np.nanmax(rgb)
    assert np.nanmax(rgb) > 0.05


def _image(sa, cam, ticks=1):
    import oracle
    return oracle_run(oracle, sa, cam, ticks=ticks)[0][-1]


def _with_layer(sa, layer, img):
    atlas = sa.atlas.copy()
    atlas[layer] = img
    return _replace(sa, atlas=atlas)


def _replace(sa, **kw):
    return dataclasses.replace(sa, **kw)


def _differs(sa, cam, sa2, what):
    assert not bits_equal(_image(sa, cam), _image(sa2, cam)), what + " does not change the oracle image"


@pytest.mark.parametrize("R", R_SIZES)
def test_materials_reach_their_branches(R):
    """metallic 1 and 0 and roughness 0 are shaded as such: nudging each changes the image.  (Roughness 0 and 1/255
    both take the 0.001 floor of the GGX terms, but not the same image: eval_specular's Smith term reads the unfloored
    roughness.)"""
    sa, cam, info = build_case("materials", R)
    for (metal, rough), new in (((255, 128), (254, 128)), ((0, 128), (1, 128)), ((128, 0), (128, 1)), ((255, 0), (255, 1))):
        img = np.empty_like(sa.atlas[0])
        img[...] = (new[0], new[1], 0, 255)
        _differs(sa, cam, _with_layer(sa, info["mr/%d/%d" % (metal, rough)], img), "metallic %d roughness %d" % (metal, rough))


@pytest.mark.parametrize("R", R_SIZES)
def test_dielectrics_reach_their_branches(R):
    """dielectric 0 takes the refraction branch (>= 0): making it -1 changes the image; ior 1 and 0.7 are shaded as
    such; the refraction cap stops paths at 0 and 1 but no path reaches 64."""
    sa, cam, _ = build_case("dielectrics", R)
    mats = sa.mats.copy()
    mats[mats[:, 10] == 0.0, 10] = -1.0
    _differs(sa, cam, _replace(sa, mats=mats), "dielectric 0")
    for ior, new in ((1.0, 1.0001), (0.7, 0.7001)):
        mats = sa.mats.copy()
        mats[mats[:, 9] == np.float32(ior), 9] = new
        _differs(sa, cam, _replace(sa, mats=mats), "ior %r" % ior)
    capped = [oracle_case("dielectrics", R, 0, cap)[2]["capped"] for cap in (0, 1, 64)]
    assert capped[0] > capped[1] > 0 and capped[2] == 0, capped


@pytest.mark.parametrize("name", ["inside_sphere", "back_quads"])
def test_inside_hits_on_non_dielectrics_grow_the_throughput(name):
    """Beer's law on inside hits of a material with a negative dielectric: 1 - (1 - diffuse) * t * dielectric > 1.
    Changing the (negative) dielectric changes the image."""
    sa, cam, _ = build_case(name, 32)
    mats = sa.mats.copy()
    neg = mats[:, 10] < 0
    assert neg.any()
    mats[neg, 10] *= 0.5
    _differs(sa, cam, _replace(sa, mats=mats), "a negative dielectric")


def test_emission_reaches_the_image():
    sa, cam, info = build_case("emission", 32)
    _differs(sa, cam, _with_layer(sa, info["emission"], np.zeros_like(sa.atlas[0])), "the emission layer")


@pytest.mark.parametrize("i", range(len(NORMAL_TEXELS)))
def test_each_normal_texel_reaches_the_image(i):
    sa, cam, info = build_case("normals", 32)
    img = sa.atlas[info["normal/%d" % i]].copy()
    img[..., 2] = 200 if img[0, 0, 2] != 200 else 100
    _differs(sa, cam, _with_layer(sa, info["normal/%d" % i], img), "normal texel %r" % (NORMAL_TEXELS[i],))


@pytest.mark.parametrize("R", R_SIZES)
def test_single_texel_layers_are_sampled_where_they_differ(R):
    """Each layer that differs from its texel 0 in one texel only is sampled there: a layer the host's constant-layer
    scan took for a colour layer would be shaded from texel 0, and replacing it by that colour changes the image.  The
    layer that differs in alpha only must not change it: the shaders never read alpha."""
    sa, cam, info = build_case("layers", R)
    for name in ("first", "last", "band", "alpha"):
        layer = sa.atlas[info["scan/" + name]]
        flat = layer.reshape(-1, 4)
        assert (flat != flat[0]).any(axis=1).sum() == (R * R - 1 if name == "first" else 1), name
        const = np.empty_like(layer)
        const[...] = flat[0]
        same = bits_equal(_image(sa, cam), _image(_with_layer(sa, info["scan/" + name], const), cam))
        assert same == (name == "alpha"), name


@pytest.mark.parametrize("R", R_SIZES)
def test_huge_uvs_are_beyond_the_guard(R):
    sa, _, _ = build_case("uvs", R)
    assert np.abs(sa.uvs).max() * R > 1e9 and np.abs(sa.uvs).max() < 1e9


@pytest.mark.parametrize("name", ["env_top", "env_bottom"])
def test_environment_rows_reach_the_image(name):
    sa, cam, _ = build_case(name, 32)
    sa2, _, _ = build_case("env_const", 32)
    assert not bits_equal(_image(sa, cam), _image(_replace(sa, env=sa2.env, bins=sa2.bins), cam))
    bright = sa.env[..., 3] > sa.env[..., 3].min()
    assert bright.any(axis=1).sum() == 1 and bright[0 if name == "env_top" else -1].all()


def test_every_stored_output_is_also_checked_on_the_cuda_path():
    """test_cuda_against_the_reference_shaders checks every record of the file, from the same case list."""
    with np.load(PATH) as z:
        stored = {k.rsplit(":", 1)[0] for k in z.files}
    assert stored == set(record_keys())


# ---------------------------------------------------------------------------------------------------------------------
# GPU
def _render(ctx, cam, sanitize, anyhit, cap, ticks=TICKS):
    ctx.set_param(capi.PARAM_SANITIZE_NAN, sanitize)
    ctx.set_param(capi.PARAM_ANYHIT, anyhit)
    ctx.set_param(capi.PARAM_MAX_REFRACTIONS, cap)
    rc, rt = scenes.rand_bases(ticks, SEED)
    capped0 = ctx.stats()["capped_paths"]
    ctx.clear()
    ctx.render(ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"]), 0, rc, rt)
    s = ctx.stats()
    s["capped"] = s["capped_paths"] - capped0
    return ctx.read_accum(), ctx.debug_last_color(), s


@pytest.mark.gpu
@pytest.mark.parametrize("plain", [False, True], ids=["interleaved", "plain"])
@pytest.mark.parametrize("name,R", IDS)
def test_cuda_against_the_oracle(name, R, plain, monkeypatch):
    """Accumulator (RGBA), last sample colour, rays, node and leaf visits and capped paths, bit for bit / exactly, with
    NaN sanitising on and off, any-hit on and off, and each refraction cap of the case; plain = k_shade<false> on the
    RGBA8 layered atlas, interleaved = k_shade<true> on the per-material atlas."""
    if plain:
        monkeypatch.setenv("FSPT_PLAIN_ATLAS", "1")
    sa, cam, _ = build_case(name, R)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        for cap in CAPS.get(name, (64,)):
            for sanitize in (0, 1):
                fbs, col, tot = oracle_case(name, R, sanitize, cap)
                for anyhit in (0, 1):
                    what = "%s R%d %s cap %d sanitize %d any-hit %d" % (name, R, "plain" if plain else "interleaved",
                                                                       cap, sanitize, anyhit)
                    fb, last, s = _render(ctx, cam, sanitize, anyhit, cap)
                    assert_bit_equal(fb, fbs[-1], what + ": accumulator")
                    assert_bit_equal(last[..., :3], col[..., :3], what + ": last sample colour")
                    assert s["last_rays"] == tot["rays"] and s["capped"] == tot["capped"], (what, s, tot)
                    if anyhit:  # hit-or-miss rays of the last bounce may stop at their first intersection
                        assert s["last_node_visits"] <= tot["node_visits"] and s["last_leaf_visits"] <= tot["leaf_visits"]
                    else:
                        assert (s["last_node_visits"], s["last_leaf_visits"]) == (tot["node_visits"], tot["leaf_visits"]), what
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("plain", [False, True], ids=["interleaved", "plain"])
@pytest.mark.parametrize("name,R", IDS)
def test_cuda_against_the_reference_shaders(name, R, plain, monkeypatch):
    """No oracle in between: the accumulator after every tick against tracer.fs's, without NaN sanitising and with no
    effective refraction cap, like the reference."""
    if plain:
        monkeypatch.setenv("FSPT_PLAIN_ATLAS", "1")
    sa, cam, _ = build_case(name, R)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        for k in range(1, TICKS + 1):
            fb, _, _ = _render(ctx, cam, 0, 1, CUDA_UNCAPPED, ticks=k)
            golden.check(record_key(name, R, k - 1), fb, path=PATH)
    finally:
        ctx.close()
