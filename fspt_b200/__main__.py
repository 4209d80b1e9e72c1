"""Headless front end: `python -m fspt_b200 <scene.json | bunny | soup | pbr> --res 1280x720 --spp 256 -o out.png`.
The URL parameters of the reference page (`?scene=..&res=WxH`, main.js:953-973) become CLI flags; the render loop is
main.js tick() (`max+1` samples, :841) and the PNG is what `canvas.toBlob` would upload (:861)."""
import argparse
import time

import numpy as np


def main():
    ap = argparse.ArgumentParser(prog="python -m fspt_b200")
    ap.add_argument("scene", help="path to a scene JSON, or one of the built-in procedural scenes: bunny, soup, pbr")
    ap.add_argument("--res", default="1280x720")
    ap.add_argument("--spp", type=int, default=None, help="samples per pixel (default: scene.samples + 1, like the reference); "
                    "with --max-rel-error, the most any pixel gets")
    ap.add_argument("--max-rel-error", type=float, default=None,
                    help="adaptive sampling: stop a pixel once the relative standard error of its mean luminance is below this")
    ap.add_argument("--min-spp", type=int, default=16, help="adaptive sampling: samples every pixel gets first (>= 2)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--denoise", action="store_true")
    ap.add_argument("--exposure", type=float, default=None)
    ap.add_argument("--saturation", type=float, default=1.0)
    ap.add_argument("--mode", default="", help="'test' = bvh_test.fs visit-count heat map (main.js:882-884)")
    ap.add_argument("-o", "--output", default="out.png")
    a = ap.parse_args()
    from . import scenes
    from .path_tracer import PathTracer
    W, H = [int(x) for x in a.res.lower().split("x")]
    t0 = time.time()
    if a.scene in ("bunny", "soup", "pbr"):
        sa, cam = {"bunny": scenes.bunny_class, "soup": scenes.sphere_soup, "pbr": scenes.pbr_scene}[a.scene](device=a.device)
        pt = PathTracer(sa, (W, H), cam, device=a.device, seed=a.seed)
    else:
        pt = PathTracer.from_scene(a.scene, (W, H), device=a.device, seed=a.seed)
    if a.exposure is not None:
        pt.exposure = a.exposure
    pt.saturation, pt.denoise = a.saturation, a.denoise
    print("scene compiled + uploaded in %.1f s: %d triangles, %d BVH nodes" % (time.time() - t0, pt.scene.n_tris, pt.scene.bvh.shape[0]))
    from PIL import Image
    if a.mode == "test":
        fr = pt._frame()
        _, _, cnt, _, _ = pt.ctx.debug_primary(fr, 1234.5, want_rays=False)
        heat = np.clip(cnt.reshape(H, W).astype(np.float32) * 0.001, 0, 1)  # bvh_test.fs:230
        Image.fromarray((heat[::-1] ** 0.4545 * 255).astype(np.uint8)).save(a.output)
        print("visit-count heat map ->", a.output)
        return
    spp = a.spp if a.spp is not None else pt.maxSamples + 1
    t0 = time.time()
    if a.max_rel_error is not None:
        pt.converge(a.max_rel_error, max_samples=spp, min_samples=a.min_spp)
    else:
        pt.tick(spp)
    img = pt.image()
    dt = time.time() - t0
    st = pt.stats()
    Image.fromarray(np.ascontiguousarray(img)).save(a.output)
    print("%d spp in %.2f s: %.1f Mpath-samples/s, %.1f Mrays/s, %.1f samples per pixel on average -> %s"
          % (spp, dt, st["samples"] / dt / 1e6, st["rays"] / dt / 1e6, st["samples"] / (W * H), a.output))


if __name__ == "__main__":
    main()
