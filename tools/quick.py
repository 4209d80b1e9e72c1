#!/usr/bin/env python
"""Quick A/B harness for kernel work: renders the bench scene for a few spp and prints per-kernel-class times."""
import argparse, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from fspt_b200 import scenes
from fspt_b200.path_tracer import PathTracer

ap = argparse.ArgumentParser()
ap.add_argument("--spp", type=int, default=16)
ap.add_argument("--scene", default="bunny")
ap.add_argument("--res", default="1280x720")
ap.add_argument("--reps", type=int, default=3)
a = ap.parse_args()
W, H = [int(x) for x in a.res.split("x")]
if a.scene == "bunny":
    sa, cam = scenes.bunny_class(subdiv=6, atlas_res=2048)
elif a.scene == "soup":
    sa, cam = scenes.sphere_soup()
elif a.scene == "pbr":
    sa, cam = scenes.pbr_scene()
elif a.scene == "soup10m":
    t0 = time.time()
    sa, cam = scenes.sphere_soup(subdiv=8, n_soup=10000000 - 1310720, seed=4321)
    print("compiled %d tris, %d nodes, depth %d in %.1f s" % (sa.n_tris, sa.bvh.shape[0], sa.depth, time.time() - t0))
pt = PathTracer(sa, (W, H), cam)
rc, rt = scenes.rand_bases(a.spp, 1)
for r in range(a.reps + 1):
    pt.clear()
    pt.tick(a.spp, rc, rt)
    st = pt.stats()
    if r:
        import zlib
        crc = zlib.crc32(pt.accumulation().tobytes())
        n = W * H * a.spp
        # trace and shade are summed launch times; the two row bands of a wave overlap, so "overlap" = how much their
        # sum exceeds the render (negative: time outside those launches -- accumulation, small launches, gaps)
        print("render %.2f ms  trace %.2f  shade %.2f  overlap %.2f | %.1f Mpaths/s %.1f Mrays/s | V/ray %.1f L/ray %.2f | crc %08x" % (
            st["render_ms"], st["trace_ms"], st["shade_ms"], st["trace_ms"] + st["shade_ms"] - st["render_ms"],
            n / st["render_ms"] / 1e3, st["last_rays"] / st["render_ms"] / 1e3,
            st["last_node_visits"] / st["last_rays"], st["last_leaf_visits"] / st["last_rays"], crc))
