#!/usr/bin/env python
"""A/B harness for kernel knobs: builds one library variant per `name:-DFLAG=..,-DFLAG2=..` argument under
fspt_b200/lib/variants/ (they travel to the GPU box with the snapshot) and prints the gpurun command that times the
default build and every variant with tools/quick.py.

  python tools/ab.py r16:-DTRACE_REFILL=16 st8:-DTRACE_SMEM_STACK=8 --scenes bunny soup
"""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fspt_b200 import build

ap = argparse.ArgumentParser()
ap.add_argument("variants", nargs="+", help="name:-DA=1,-DB=2")
ap.add_argument("--scenes", nargs="+", default=["bunny"])
ap.add_argument("--spp", type=int, default=64)
a = ap.parse_args()
names = []
for v in a.variants:
    name, _, flags = v.partition(":")
    out = build.build(defines=[f for f in flags.split(",") if f], out="lib/variants/%s.so" % name)
    print("built", out)
    names.append(name)
loop = " ".join(['""'] + names)
print("\n/usr/local/graft/bin/gpurun --timeout 900 -- 'for v in %s; do echo \"== $v\"; for s in %s; do "
      "FSPT_LIB=${v:+fspt_b200/lib/variants/$v.so} python tools/quick.py --scene $s --reps 2 --spp %d 2>&1 | tail -1; "
      "done; done'" % (loop, " ".join(a.scenes), a.spp))
