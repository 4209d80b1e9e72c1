"""Measure the FSPT-DM2 built-ins (oracle/oracle_math.h) against float64 libm, exhaustively.

Every f32 input of each range below is evaluated by the oracle and compared with numpy's float64 function; atan2 is
measured over V x V (oracle/dm_edges.py, finite pairs).  An ulp is the spacing of the float64 reference rounded to f32
(as tests/test_oracle_cpu.py::test_dm_math_is_faithful measures it).  Prints each worst case and its argument; these are
the bounds DESIGN.md section 2 states.  CPU only: `python tools/dm_accuracy.py [--only sin,log2]` (about a minute per
function on 8 cores).
"""
import argparse
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle  # noqa: E402
from oracle import dm_edges  # noqa: E402

CHUNK = 1 << 24
GAMMA = np.float32(0.454545)  # draw.fs's gamma exponent


def bits(v):
    return int(np.float32(v).view(np.uint32))


def ulps(got, ref64):
    return np.abs(got.astype(np.float64) - ref64) / np.maximum(np.spacing(np.abs(ref64.astype(np.float32))).astype(np.float64), 1e-45)


# name -> (probe, float64 reference, inclusive bit ranges, [(metric name, mask(x) or None, error(got, ref64, x))])
def _ulp(mask=None):
    return ("ulp", mask, lambda g, r, x: ulps(g, r))


def _abs(mask=None):
    return ("abs", mask, lambda g, r, x: np.abs(g.astype(np.float64) - r))


NEG = 0x80000000
MEASURES = {
    "sin": ("sin", np.sin, [(0, bits(1e7)), (NEG, NEG | bits(1e7))],
            [("ulp |x| <= 64", lambda x: np.abs(x) <= 64, lambda g, r, x: ulps(g, r)), ("abs |x| <= 1e7",) + _abs()[1:]]),
    "cos": ("cos", np.cos, [(0, bits(1e7)), (NEG, NEG | bits(1e7))],
            [("ulp |x| <= 64", lambda x: np.abs(x) <= 64, lambda g, r, x: ulps(g, r)), ("abs |x| <= 1e7",) + _abs()[1:]]),
    "asin": ("asin", np.arcsin, [(0, bits(1.0)), (NEG, NEG | bits(1.0))], [("ulp |x| <= 1",) + _ulp()[1:]]),
    "exp2": ("exp2", np.exp2, [(0, bits(127.0)), (NEG, NEG | bits(126.0))], [("ulp [-126, 127]",) + _ulp()[1:]]),
    "log2": ("log2", np.log2, [(1, 0x7F7FFFFF)], [("ulp x > 0 finite",) + _ulp()[1:]]),
    "gamma": ("pow", lambda x: np.power(x, np.float64(GAMMA)), [(0, bits(1.0))],
              [("8-bit steps, x in [0, 1]", None, lambda g, r, x: np.abs(g.astype(np.float64) - r) * 255)]),
}


def run(name, pool):
    probe, ref, ranges, metrics = MEASURES[name]
    worst = [(0.0, None)] * len(metrics)
    y = GAMMA if name == "gamma" else None

    def chunk(a, b):
        x = np.arange(a, b, dtype=np.uint32).view(np.float32)
        g = oracle.dm_eval(probe, x, None if y is None else np.full_like(x, y))
        r = ref(x.astype(np.float64))
        out = []
        for _, mask, err in metrics:
            e = err(g, r, x)
            if mask is not None:
                e = np.where(mask(x), e, 0.0)
            i = int(np.argmax(e))
            out.append((float(e[i]), x[i]))
        return out
    futs = [pool.submit(chunk, a, min(a + CHUNK, hi + 1)) for lo, hi in ranges for a in range(lo, hi + 1, CHUNK)]
    for f in futs:
        for k, (e, x) in enumerate(f.result()):
            if e > worst[k][0]:
                worst[k] = (e, x)
    return [(m[0], e, x) for m, (e, x) in zip(metrics, worst)]


def atan2_edges():
    V = dm_edges.values()
    V = V[np.isfinite(V)]
    x, y = np.repeat(V, V.size), np.tile(V, V.size)
    # y = +-0: the model ignores the zero's sign (atan2(-0, x < 0) = +pi, atan2(0, 0) = 0), libm does not
    keep = y != 0
    rng = np.random.default_rng(0)  # and uniform pairs on [-1, 1]^2, where the shaders' directions lie
    u, v = rng.uniform(-1, 1, 1 << 24).astype(np.float32), rng.uniform(-1, 1, 1 << 24).astype(np.float32)
    rows = []
    for what, (a, b) in (("ulp, finite V x V, y != 0", (x[keep], y[keep])), ("ulp, 2^24 uniform [-1, 1]^2", (u, v))):
        e = ulps(oracle.dm_eval("atan2", a, b), np.arctan2(b.astype(np.float64), a.astype(np.float64)))
        i = int(np.argmax(e))
        rows.append((what, float(e[i]), (b[i], a[i])))
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--only", default="", help="comma-separated subset of: " + ", ".join(list(MEASURES) + ["atan2"]))
    args = ap.parse_args()
    names = args.only.split(",") if args.only else list(MEASURES) + ["atan2"]
    with ThreadPoolExecutor(os.cpu_count() or 1) as pool:
        for name in names:
            t0 = time.perf_counter()
            rows = atan2_edges() if name == "atan2" else run(name, pool)
            for metric, e, x in rows:
                at = "(y, x) = (%s, %s)" % (float(x[0]).hex(), float(x[1]).hex()) if isinstance(x, tuple) else \
                    "x = %s (%.9g)" % (float(x).hex(), x)
                print("%-6s %-26s worst %.4g at %s   [%.0f s]" % (name, metric, e, at, time.perf_counter() - t0), flush=True)


if __name__ == "__main__":
    main()
