"""Wall-clock time of the two BVH builders on the same inputs: the host builder (fspt_bvh_build2, every host thread) and
the device builder (fspt_bvh_build_device, upload and download included).  Each call returns synchronised, so the clock
around it is the time a caller waits.  The builders alternate on every input, after a warm-up, and every result is
checked bit for bit against the other builder's.  Prints the card and its power limit first.

  python tools/bvh_time.py [--reps 3] [--max-tris 10000000] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fspt_b200 import capi, procedural as pr, scenes  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError as e:
        return "nvidia-smi unavailable (%s)" % e


def inputs(max_tris):
    yield "config3", lambda: scenes.sphere_soup_verts()
    if max_tris >= 10000000:
        yield "config5", lambda: scenes.sphere_soup_verts(subdiv=8, n_soup=10000000 - 1310720, seed=4321)
    T = 1000
    while T <= max_tris:
        yield "soup%d" % T, (lambda T=T: pr.triangle_soup(T, 4321).reshape(-1, 9))
        T *= 10


def timed(fn, *a, **k):
    t0 = time.perf_counter()
    r = fn(*a, **k)
    return (time.perf_counter() - t0) * 1e3, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-tris", type=int, default=10000000)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not capi.device_usable(a.device):
        sys.exit("no usable sm_100 device: %s" % capi.load().fspt_last_error(None).decode())
    print("card: %s | host threads: %d" % (card(), os.cpu_count()), flush=True)
    warm = pr.triangle_soup(20000, 1).reshape(-1, 9)
    capi.bvh_build(warm)
    capi.bvh_build_device(warm, device=a.device)
    rows = []
    for name, make in inputs(a.max_tris):
        v = make()
        host_ms, dev_ms = [], []
        for _ in range(a.reps):
            th, h = timed(capi.bvh_build, v)
            td, d = timed(capi.bvh_build_device, v, device=a.device)
            assert np.array_equal(h[0].view(np.uint32), d[0].view(np.uint32)) and np.array_equal(h[1], d[1]) and h[2] == d[2], \
                "%s: the builders disagree" % name
            host_ms.append(th)
            dev_ms.append(td)
        row = dict(input=name, triangles=int(v.shape[0]), nodes=int(h[0].shape[0]), depth=h[2],
                   host_ms=sorted(host_ms), device_ms=sorted(dev_ms))
        rows.append(row)
        print("%-14s T=%9d  host %9.1f ms  device %8.1f ms  (median of %d; min %.1f / %.1f)  x%.1f  identical" % (
            name, row["triangles"], np.median(host_ms), np.median(dev_ms), a.reps, min(host_ms), min(dev_ms),
            np.median(host_ms) / np.median(dev_ms)), flush=True)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(dict(card=card(), host_threads=os.cpu_count(), rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
