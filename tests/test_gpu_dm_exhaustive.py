"""The device's scalar arithmetic against the oracle's, bit for bit, over the whole binary32 range.

Every bit-exact render test rests on dm_math.cuh / device_common.cuh computing what oracle_math.h / oracle_texunit.h
compute for every input, not only for the arguments the scenes happen to produce.  Unary probes run on all 2^32 bit
patterns; binary probes on V x V, V being oracle/dm_edges.py's structured set (every exponent, every branch edge of the
model +-2 ulp, the shared-reciprocal division's window).  A NaN matches any NaN (the model does not fix payloads); the
int-valued probe is compared bit for bit.  The slab test's packed f32x2 subtraction and multiplication (FADD2 / FMUL2
with a broadcast scalar operand) are compared on both lanes with numpy's float32 arithmetic, which is correctly rounded
IEEE: a packed pipe that flushed subnormals or treated inf / NaN differently would change box order and visit counts.
The file takes about 4 minutes on a B200 host."""
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import dm_edges

CHUNK = 1 << 26
THREADS = max(1, min(32, os.cpu_count() or 1))
# probe -> the oracle's answers it is compared with (sincos: both outputs of one call)
UNARY = {"sin": ("sin",), "cos": ("cos",), "sincos": ("sincos_s", "sincos_c"), "asin": ("asin",), "exp2": ("exp2",),
         "log2": ("log2",), "rnd": ("rnd",), "clamp": ("clamp",), "coord_to_i32": ("coord_to_i32",), "quant8": ("quant8",)}
BINARY = ("atan2", "pow", "min", "max", "div", "div_shared", "div_z")
# slab_pair's packed lanes: (x, -x) against the broadcast y
PACKED = {"sub2_lo": lambda x, y: x - y, "sub2_hi": lambda x, y: -x - y, "mul2_lo": lambda x, y: x * y,
          "mul2_hi": lambda x, y: -x * y}
INT_BITS = {"coord_to_i32"}  # the output holds an int's bits, some of which read as NaN: compare bits exactly


def _mismatch(got, ref, exact):
    bad = got.view(np.uint32) != ref.view(np.uint32)
    if not exact:
        bad &= ~(np.isnan(got) & np.isnan(ref))
    return np.flatnonzero(bad)


def _report(fn, idx, got, ref, x, y=None):
    i = idx[0]
    args = "x=0x%08x" % x.view(np.uint32)[i] + ("" if y is None else " y=0x%08x" % y.view(np.uint32)[i])
    return "%s: %d mismatches; first at %s (%r%s): device 0x%08x, oracle 0x%08x" % (
        fn, idx.size, args, x[i], "" if y is None else ", %r" % y[i], got.view(np.uint32)[i], ref.view(np.uint32)[i])


def _oracle(pool, oracle_mod, fn, x, y=None):
    """oracle.dm_eval over x (and y) in THREADS slices at once (ctypes releases the GIL); returns a future-like."""
    out = np.empty_like(x)
    bounds = np.linspace(0, x.size, THREADS + 1).astype(np.int64)

    def part(a, b):
        out[a:b] = oracle_mod.dm_eval(fn, x[a:b], None if y is None else y[a:b])
    futs = [pool.submit(part, a, b) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
    return lambda: ([f.result() for f in futs], out)[1]


@pytest.fixture(scope="module")
def ctx():
    from fspt_b200 import capi
    c = capi.Context(8, 8)
    yield c
    c.close()


@pytest.fixture(scope="module")
def pool():
    with ThreadPoolExecutor(THREADS) as p:
        yield p


@pytest.mark.gpu
@pytest.mark.parametrize("fn", list(UNARY))
def test_unary_every_f32(ctx, oracle_mod, pool, fn):
    t0 = time.perf_counter()
    for c in range((1 << 32) // CHUNK):
        x = np.arange(c * CHUNK, (c + 1) * CHUNK, dtype=np.uint32).view(np.float32)
        refs = [_oracle(pool, oracle_mod, name, x) for name in UNARY[fn]]  # the oracle works while the device does
        for name, ref in zip(UNARY[fn], refs):
            got = ctx.debug_math(name, x)
            ref = ref()
            idx = _mismatch(got, ref, fn in INT_BITS)
            assert idx.size == 0, _report(name, idx, got, ref, x)
    print("%s: 2^32 inputs in %.1f s" % (fn, time.perf_counter() - t0))


@pytest.mark.gpu
@pytest.mark.parametrize("fn", BINARY)
def test_binary_edges(ctx, oracle_mod, pool, fn):
    V = dm_edges.values()
    x, y = np.repeat(V, V.size), np.tile(V, V.size)
    ref = _oracle(pool, oracle_mod, fn, x, y)
    got = ctx.debug_math(fn, x, y)
    ref = ref()
    idx = _mismatch(got, ref, False)
    assert idx.size == 0, _report(fn, idx, got, ref, x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("fn", list(PACKED))
def test_packed_slab_arithmetic_edges(ctx, oracle_mod, fn):
    V = dm_edges.values()
    x, y = np.repeat(V, V.size), np.tile(V, V.size)
    with np.errstate(all="ignore"):
        ref = PACKED[fn](x, y)
    for who, got in (("device", ctx.debug_math(fn, x, y)), ("oracle", oracle_mod.dm_eval(fn, x, y))):
        idx = _mismatch(got, ref, False)
        assert idx.size == 0, who + " " + _report(fn, idx, got, ref, x, y)


def test_packed_probe_operands_reach_every_class():
    """V x V gives the packed lanes subnormal and overflowing results and every inf / NaN operand pairing"""
    V = dm_edges.values()
    x, y = np.repeat(V, V.size), np.tile(V, V.size)
    tiny = np.finfo(np.float32).tiny
    with np.errstate(all="ignore"):
        for f in PACKED.values():
            r = f(x, y)
            fin = np.isfinite(x) & np.isfinite(y)
            assert ((r != 0) & (np.abs(r) < tiny)).sum() > 1000 and np.isinf(r[fin]).sum() > 1000 and np.isnan(r).any()


@pytest.mark.gpu
def test_debug_math_rejects_unknown_code(ctx):
    from fspt_b200 import capi
    for code in (-1, len(capi.DEBUG_MATH), 1 << 20):
        with pytest.raises(capi.FsptError):
            ctx.debug_math(code, [1.0])


def test_probe_names_agree(oracle_mod):
    """Both sides answer the same probe names with the same codes, and the oracle refuses an unknown code."""
    from fspt_b200 import capi
    assert oracle_mod.DM_CODES == capi.DEBUG_MATH
    assert {name for names in UNARY.values() for name in names} | set(BINARY) == set(capi.DEBUG_MATH)  # each one tested
    assert oracle_mod.lib().oracle_dm_eval(len(capi.DEBUG_MATH), None, None, None, 0) == -1


def test_packed_probe_names_agree(oracle_mod):
    """Both sides answer the packed-lane probes with the same codes, apart from the scalar ones; each one is tested and
    the oracle refuses the codes around their block."""
    from fspt_b200 import capi
    assert oracle_mod.DM_PACKED_CODES == capi.DEBUG_MATH_PACKED and set(PACKED) == set(capi.DEBUG_MATH_PACKED)
    assert not set(capi.DEBUG_MATH_PACKED.values()) & set(capi.DEBUG_MATH.values())
    lo, hi = min(capi.DEBUG_MATH_PACKED.values()), max(capi.DEBUG_MATH_PACKED.values())
    assert hi - lo + 1 == len(capi.DEBUG_MATH_PACKED)
    for code in (len(capi.DEBUG_MATH), lo - 1, hi + 1):
        assert oracle_mod.lib().oracle_dm_eval(code, None, None, None, 0) == -1


@pytest.mark.gpu
def test_debug_math_rejects_codes_around_the_packed_block(ctx):
    from fspt_b200 import capi
    lo, hi = min(capi.DEBUG_MATH_PACKED.values()), max(capi.DEBUG_MATH_PACKED.values())
    for code in (len(capi.DEBUG_MATH), lo - 1, hi + 1):
        with pytest.raises(capi.FsptError):
            ctx.debug_math(code, [1.0])


def test_edge_set_holds_every_edge():
    """V holds every operand class and branch edge the binary comparisons are meant to reach."""
    V = dm_edges.values()
    b = V.view(np.uint32).astype(np.int64)
    have = set(b.tolist())
    assert V.size == len(have) and V.size < 4000  # V x V stays a few seconds on both sides
    for sign in (0, 1 << 31):
        s = lambda m: m | sign  # noqa: E731
        assert {s(0), s(0x7F800000)} <= have
        for e in range(255):  # every exponent, subnormal leading bits included
            lo, hi = (1, 1 << 23) if e == 0 else (e << 23, (e + 1) << 23)
            assert any(lo <= (m & 0x7FFFFFFF) < hi for m in (b[(b & (1 << 31)) == sign]).tolist()), (sign, e)
        for lead in range(23):
            assert s(1 << lead) in have
        for e in range(1, 255):
            assert {s(e << 23), s((e << 23) + 1), s((e << 23) + 0x7FFFFF)} <= have
        for v in dm_edges.edge_values():
            c = int(np.float32(v).view(np.uint32))
            assert {s(c + d) for d in range(-2, 3) if c + d <= 0x7F800000} <= have, float(v)
        for w in dm_edges.WINDOW:
            c = int(w.view(np.uint32))
            assert {s(c + d) for d in range(-dm_edges.WINDOW_RUN, dm_edges.WINDOW_RUN + 1)} <= have
    assert set(dm_edges.NANS) <= have and int(np.isnan(V).sum()) == 2
    # the named edges are the model's own constants
    f = np.float32
    assert dm_edges.EDGES["atan01 reduction about tan(pi/8)"] == f(0.4142135679721832)
    assert dm_edges.EDGES["log2 mantissa split"] == f(1.4142135381698608)
    assert dm_edges.EDGES["smallest normal (log2 subnormal test, div_z's ordinary divisor)"] == np.finfo(np.float32).tiny
    assert dm_edges.EDGES["largest finite (div_z's ordinary divisor)"] == np.finfo(np.float32).max
    assert dm_edges.EDGES["pow's large-x exit"] == f(3.0e38) and dm_edges.EDGES["sin/cos reduction guard and float->int guard"] == f(1e9)
    # the exp2 clamps are reached through pow: x = 2, 1/2, 4, 16 are in V, and y * log2(x) hits 130 and -160 exactly
    for x, ys in ((2.0, (130.0, -160.0)), (0.5, (-130.0, 160.0)), (4.0, (65.0, -80.0)), (16.0, (32.5, -40.0))):
        assert f(x) in V and all(f(yv) in V for yv in ys)
    # rint ties: exp2 half-integers and reduction arguments whose f32 product with 2/pi is m + 1/2
    ties = dm_edges.reduce_ties()
    assert len(ties) >= 8 and all(float(t * f(float.fromhex("0x1.45f306p-1"))) % 1.0 == 0.5 for t in ties)
    assert all(t in V and -t in V for t in ties + dm_edges.EXP2_TIES)
