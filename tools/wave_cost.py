#!/usr/bin/env python
"""Fixed cost of a render wave on the bench.py config-2 workload (bunny-class scene, 1280x720, 64 spp).

One context per samples-per-wave value S (FSPT_WAVE_SAMPLES is read when a context is created) renders the same
64 samples in turns, L2 flushed before each render like bench.py does.  A 64-sample render at S samples per wave runs
64/S waves, so the device time is fitted as T(S) = (64/S) * F + V: F is what one wave costs whatever its size (launch
ramps and tails, the per-wave small launches), V the per-path work.  Then one render at the default S is traced with
torch.profiler and every kernel is listed with its duration and the idle gap before it.

  python tools/wave_cost.py [--rounds 6] [--waves 8,16,32,64] [--out wave_cost.json]
"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from fspt_b200 import scenes
from fspt_b200.path_tracer import PathTracer

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=6)
ap.add_argument("--waves", default="8,16,32,64")
ap.add_argument("--spp", type=int, default=64)
ap.add_argument("--res", default="1280x720")
ap.add_argument("--out", default=None)
a = ap.parse_args()
W, H = [int(x) for x in a.res.split("x")]

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print("card:", card)
sa, cam = scenes.bunny_class(subdiv=6, atlas_res=2048, env_size=(2048, 1024))
rc, rt = scenes.rand_bases(a.spp, 1)
waves = [int(s) for s in a.waves.split(",")]
pts = {}
for s in waves:
    os.environ["FSPT_WAVE_SAMPLES"] = str(s)
    pts[s] = PathTracer(sa, (W, H), cam)
os.environ.pop("FSPT_WAVE_SAMPLES")
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")


def render(pt):
    flush.fill_(1)
    torch.cuda.synchronize()
    pt.clear()
    pt.tick(a.spp, rc, rt)
    return pt.stats()


times = {s: [] for s in waves}
ref = None
for r in range(a.rounds + 1):
    for s in waves:
        st = render(pts[s])
        if r:
            times[s].append(st["render_ms"])
        acc = pts[s].accumulation()
        if ref is None:
            ref = acc
        assert np.array_equal(acc.view(np.uint32), ref.view(np.uint32)), "S=%d changed the image" % s
x = np.array([a.spp / s for s in waves for _ in times[s]])
y = np.array([t for s in waves for t in times[s]])
F, V = np.polyfit(x, y, 1)
for s in waves:
    t = np.array(times[s])
    print("S=%2d  waves=%2d  render_ms mean %.3f  min %.3f  max %.3f" % (s, a.spp // s, t.mean(), t.min(), t.max()))
t64 = float(np.mean(times[max(waves)]))
print("fit T(S) = (%d/S) * F + V:  F = %.3f ms per wave, V = %.3f ms;  F / T(S=%d) = %.2f %%" % (
    a.spp, F, V, max(waves), 100 * F / t64))

# one render at the default samples per wave, every kernel with its duration and the idle gap before it
for p in pts.values():
    p.close()
pt = PathTracer(sa, (W, H), cam)
render(pt)
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    render(pt)
evs = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and
              e.name.startswith(("k_", "void k_"))], key=lambda e: e.time_range.start)
launches, prev_end, busy = [], None, 0.0
for e in evs:
    t0, t1 = e.time_range.start, e.time_range.end
    gap = (t0 - prev_end) if prev_end is not None else 0.0
    launches.append(dict(name=e.name.split("(")[0].replace("void ", ""), start_us=t0 - evs[0].time_range.start,
                         dur_us=t1 - t0, gap_before_us=gap))
    prev_end = t1 if prev_end is None else max(prev_end, t1)
    busy += t1 - t0
for L in launches:
    print("%-40s start %9.1f us  dur %9.1f us  gap before %6.1f us" % (L["name"][:40], L["start_us"], L["dur_us"],
                                                                     L["gap_before_us"]))
span = prev_end - evs[0].time_range.start if evs else 0.0
print("kernels: %d, span %.1f us, sum of kernel times %.1f us" % (len(launches), span, busy))
pt.close()
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(dict(card=card, times_ms={str(s): times[s] for s in waves}, F_ms=F, V_ms=V, t64_ms=t64,
                       launches=launches), f, indent=1)
