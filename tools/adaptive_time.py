#!/usr/bin/env python
"""Adaptive sampling (PathTracer.converge) against uniform sampling, on two scenes at 1280x720: bench.py config 2
(bunny-class) and the textured PBR scene with its refractive prop (config 4's scene).

For each threshold, an adaptive render capped at --cap samples per pixel reports its wall time (host clock around the
render and drawQuad, which ends in a synchronise), its total path samples, and the RMSE of its tonemapped RGBA8 image
against a uniform render at 4 x the cap.  Uniform renders at the cap and at the same total samples as each adaptive
render are reported the same way.  Each timing is the median of --repeat runs after one warm-up.

  python tools/adaptive_time.py [--cap 64] [--errors 0.1,0.05,0.02] [--min-spp 16] [--out adaptive_time.json]
"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from fspt_b200 import scenes
from fspt_b200.path_tracer import PathTracer

ap = argparse.ArgumentParser()
ap.add_argument("--cap", type=int, default=64)
ap.add_argument("--errors", default="0.1,0.05,0.02")
ap.add_argument("--min-spp", type=int, default=16)
ap.add_argument("--batch", type=int, default=16)
ap.add_argument("--repeat", type=int, default=3)
ap.add_argument("--res", default="1280x720")
ap.add_argument("--out", default=None)
a = ap.parse_args()
W, H = [int(x) for x in a.res.split("x")]
errors = [float(e) for e in a.errors.split(",")]

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print("card:", card)


def rmse(img, ref):
    d = img[..., :3].astype(np.float64) - ref[..., :3].astype(np.float64)
    return float(np.sqrt(np.mean(d * d)))


def timed(fn):
    fn()  # warm-up
    ts = []
    for _ in range(a.repeat):
        t0 = time.perf_counter()
        img = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), img


def uniform(pt, spp):
    def run():
        pt.ctx.set_adaptive(0, 2)
        pt.clear()
        pt.ctx.set_accum_mode(1)
        pt.tick(spp)
        return pt.drawQuad()
    return run


results = []
for name, make in (("config 2 bunny-class", lambda: scenes.bunny_class(subdiv=6, atlas_res=2048, env_size=(2048, 1024))),
                   ("PBR scene, refractive prop", lambda: scenes.pbr_scene(atlas_res=2048))):
    sa, cam = make()
    pt = PathTracer(sa, (W, H), cam)
    pt.ctx.set_accum_mode(1)
    ref_spp = 4 * a.cap
    pt.clear()
    pt.tick(ref_spp)
    ref = pt.drawQuad().copy()
    rows = []
    t, img = timed(uniform(pt, a.cap))
    rows.append(dict(kind="uniform", spp=a.cap, samples=W * H * a.cap, seconds=t, rmse=rmse(img, ref)))
    for err in errors:
        def run(err=err):
            return pt.converge(err, max_samples=a.cap, min_samples=a.min_spp, batch=a.batch)
        t, img = timed(run)
        samples = int(pt.stats()["samples"])
        rows.append(dict(kind="adaptive", max_rel_error=err, spp=a.cap, samples=samples, seconds=t, rmse=rmse(img, ref)))
        spp_eq = max(1, int(round(samples / (W * H))))
        t, img = timed(uniform(pt, spp_eq))
        rows.append(dict(kind="uniform, equal samples", spp=spp_eq, samples=W * H * spp_eq, seconds=t, rmse=rmse(img, ref)))
    pt.close()
    print("%s, %dx%d, reference: uniform %d spp" % (name, W, H, ref_spp))
    for r in rows:
        label = r["kind"] + (" %.3g" % r["max_rel_error"] if "max_rel_error" in r else "")
        print("  %-28s spp<=%4d  samples %11d (%.1f per pixel)  %.3f s  RMSE %.3f" % (
            label, r["spp"], r["samples"], r["samples"] / (W * H), r["seconds"], r["rmse"]))
    results.append(dict(scene=name, reference_spp=ref_spp, rows=rows))
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(dict(card=card, res=[W, H], cap=a.cap, min_spp=a.min_spp, batch=a.batch, results=results), f, indent=1)
