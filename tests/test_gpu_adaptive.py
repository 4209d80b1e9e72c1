"""Adaptive sampling in sum mode (fspt_set_adaptive).  A pixel's samples do not depend on which pixels are rendered with
it, and a pixel that stops keeps its statistics, so a pixel that received n ticks must equal, bit for bit, the uniform
sum-mode render after n ticks -- accumulator, moment and last sample colour.  Adaptive renders run in calls of `batch`
ticks with slices of the rand bases, as a uniform render would.  The rule is restated here in numpy f32, in the order the
header gives, and must select exactly the pixels the library renders."""
import os
import re

import numpy as np
import pytest

from fspt_b200 import capi, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

LC = np.float32([0.2126, 0.7152, 0.0722])  # draw.fs lumaCoefs
FLOOR = np.float32(1e-3)


def _frame(ctx, cam):
    return ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])


def _luma(c):
    return (c[..., 0] * LC[0] + c[..., 1] * LC[1]) + c[..., 2] * LC[2]


def _rule(acc, m2, err, min_s):
    """The selection rule of fspt_set_adaptive, every step in f32, in the header's order."""
    n = acc[..., 3]
    with np.errstate(all="ignore"):
        mean = _luma(acc) / n
        var = (m2 / n - mean * mean) * (n / (n - np.float32(1)))
        err_ok = np.sqrt(np.fmax(var, np.float32(0)) / n) > np.float32(err) * np.fmax(mean, FLOOR)
    return (n < np.float32(min_s)) | err_ok


def _uniform(ctx, fr, rc, rt):
    """Sum mode, one tick per call: the accumulator and the clamped sample colour after every tick, and the moment
    (numpy f32 sum of the squared luminances, in tick order) after every tick."""
    ctx.clear()
    ctx.set_accum_mode(1)
    accs, lasts = [], []
    for k in range(len(rc)):
        ctx.render(fr, k, rc[k:k + 1], rt[k:k + 1])
        accs.append(ctx.read_accum())
        lasts.append(ctx.debug_last_color())
    l = _luma(np.stack(lasts))
    m, m2s = np.zeros(l.shape[1:], np.float32), []
    for k in range(len(rc)):
        m = m + l[k] * l[k]
        m2s.append(m)
    return np.stack(accs), np.stack(lasts), np.stack(m2s)


def _wave_starts(n_ticks, batch, wave_s):
    """The ticks at which a wave starts when n_ticks are rendered in calls of `batch` with waves of wave_s samples."""
    starts = []
    for k0 in range(0, n_ticks, batch):
        n = min(batch, n_ticks - k0)
        starts += list(range(k0, k0 + n, wave_s))
    return starts


def _simulate(accs, m2s, starts, err, min_s):
    """Per pixel, the ticks it receives: the rule, applied before each wave to the uniform state after that many ticks."""
    n_ticks = accs.shape[0]
    n = np.zeros(accs.shape[1:3], np.int64)
    live = np.ones_like(n, bool)
    for b, e in zip(starts, starts[1:] + [n_ticks]):
        if b > 0:
            live &= _rule(accs[b - 1], m2s[b - 1], err, min_s)
        n[live] = e
    return n


def _adaptive(ctx, fr, rc, rt, err, min_s, batch, rects, check_rule=False):
    """Adaptive render of every rectangle in turn, in calls of `batch` ticks.  check_rule: before each call the numpy rule
    gives exactly the pixels whose count grows in the call, and active_pixels() their number."""
    ctx.clear()
    ctx.set_accum_mode(1)
    ctx.set_adaptive(err, min_s)
    for x, y, w, h in rects:
        ctx.set_tile(x, y, w, h)
        for k0 in range(0, len(rc), batch):
            if check_rule:
                acc = ctx.read_accum()
                want = np.zeros(acc.shape[:2], bool)
                want[y:y + h, x:x + w] = _rule(acc, ctx.read_moment(), err, min_s)[y:y + h, x:x + w]
                assert ctx.active_pixels() == int(want.sum()), k0
            ctx.render(fr, k0, rc[k0:k0 + batch], rt[k0:k0 + batch])
            if check_rule:
                assert np.array_equal(ctx.read_accum()[..., 3] > acc[..., 3], want), k0
    return ctx.read_accum(), ctx.read_moment()


def _check_prefix(acc, m2, last, accs, lasts, m2s, n_sim):
    """Every pixel equals the uniform render after its own count of ticks, bit for bit."""
    n = acc[..., 3].astype(np.int64)
    assert np.array_equal(n, n_sim)
    yy, xx = np.indices(n.shape)
    k = n - 1
    assert np.array_equal(acc.view(np.uint32), accs[k, yy, xx].view(np.uint32))
    assert np.array_equal(m2.view(np.uint32), m2s[k, yy, xx].view(np.uint32))
    assert np.array_equal(last.view(np.uint32), lasts[k, yy, xx].view(np.uint32))


def _pick_threshold(accs, m2s, starts, min_s):
    """A threshold that stops some pixels at min_samples and leaves others at the cap (the most balanced one)."""
    best = None
    for err in (0.5, 0.3, 0.2, 0.1, 0.05, 0.03, 0.02, 0.01, 0.005):
        n = _simulate(accs, m2s, starts, err, min_s)
        score = min((n == min_s).mean(), (n == accs.shape[0]).mean())
        if best is None or score > best[0]:
            best = (score, err, n)
    assert best[0] > 0, "no threshold stops some pixels at min_samples and leaves others at the cap"
    return best[1], best[2]


def _refractive():
    return scenes.pbr_scene(atlas_res=64, subdiv=2, env_size=(128, 64))


@gpu
@pytest.mark.parametrize("scene", ["bunny", "refractive"])
def test_stopped_pixels_equal_the_uniform_render_at_their_count(small_bunny, scene):
    sa, cam = small_bunny if scene == "bunny" else _refractive()
    W, H, N, batch, min_s = 64, 48, 24, 4, 4
    rc, rt = scenes.rand_bases(N, 31)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        accs, lasts, m2s = _uniform(ctx, fr, rc, rt)
        starts = _wave_starts(N, batch, batch)
        err, n_sim = _pick_threshold(accs, m2s, starts, min_s)
        acc, m2 = _adaptive(ctx, fr, rc, rt, err, min_s, batch, [(0, 0, W, H)], check_rule=True)
        _check_prefix(acc, m2, ctx.debug_last_color(), accs, lasts, m2s, n_sim)
        n = acc[..., 3]
        assert (n == min_s).any() and (n == N).any()
        assert ctx.stats()["samples"] == int(n.sum())
        assert ctx.accum_device_ptr()[2] == N  # the ticks, not the samples
    finally:
        ctx.close()


@gpu
@pytest.mark.parametrize("case", ["two_bands", "untiled", "tile_offsets"])
def test_rectangles_one_after_the_other_equal_the_whole(small_bunny, case):
    """The whole rectangle and the same pixels as strips or tiles, one after the other, bit for bit in the accumulator
    and the moment.  two_bands: 256 x 256 at 32 spp splits each wave into two bands, strips of 16 rows do not."""
    sa, cam = small_bunny
    W, H, N, batch, min_s, whole, parts = {
        "two_bands": (256, 256, 32, 8, 8, (0, 0, 256, 256), [(0, y, 256, 16) for y in range(0, 256, 16)]),
        "untiled": (272, 70, 12, 4, 4, (5, 3, 250, 61), [(5, y, 250, min(7, 64 - y)) for y in range(3, 64, 7)]),
        "tile_offsets": (200, 150, 12, 4, 4, (0, 0, 200, 150),
                         [(0, 0, 96, 72), (96, 0, 104, 72), (0, 72, 96, 78), (96, 72, 104, 78)]),
    }[case]
    rc, rt = scenes.rand_bases(N, 32)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        for err in (0.05, 0.02, 0.1):
            acc, m2 = _adaptive(ctx, fr, rc, rt, err, min_s, batch, [whole])
            x, y, w, h = whole
            n = acc[y:y + h, x:x + w, 3]
            if n.min() < n.max():
                break
        assert n.min() < n.max() == N, (n.min(), n.max())
        acc1, m21 = _adaptive(ctx, fr, rc, rt, err, min_s, batch, parts)
        assert np.array_equal(acc.view(np.uint32), acc1.view(np.uint32))
        assert np.array_equal(m2.view(np.uint32), m21.view(np.uint32))
        assert ctx.stats()["samples"] == int(acc[..., 3].sum())
    finally:
        ctx.close()


@gpu
def test_several_waves_per_call(small_bunny, monkeypatch):
    """3 samples per wave, calls of 7 ticks: waves of 3, 3 and 1, the first two split into two bands, the last one not.
    Pixels stop inside a call, and every stopped pixel still equals the uniform render at its count."""
    monkeypatch.setenv("FSPT_WAVE_SAMPLES", "3")
    sa, cam = small_bunny
    W, H, N, batch, min_s = 512, 384, 21, 7, 3
    rc, rt = scenes.rand_bases(N, 33)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        accs, lasts, m2s = _uniform(ctx, fr, rc, rt)
        starts = _wave_starts(N, batch, 3)
        assert starts == [0, 3, 6, 7, 10, 13, 14, 17, 20]
        err, n_sim = _pick_threshold(accs, m2s, starts, min_s)
        acc, m2 = _adaptive(ctx, fr, rc, rt, err, min_s, batch, [(0, 0, W, H)], check_rule=True)
        _check_prefix(acc, m2, ctx.debug_last_color(), accs, lasts, m2s, n_sim)
        n = acc[..., 3].astype(np.int64)
        assert ((n % batch) != 0).any() and (n == min_s).any() and (n == N).any()
        acc1, m21 = _adaptive(ctx, fr, rc, rt, err, min_s, batch, [(0, y, W, 32) for y in range(0, H, 32)])
        assert np.array_equal(acc.view(np.uint32), acc1.view(np.uint32))
        assert np.array_equal(m2.view(np.uint32), m21.view(np.uint32))
    finally:
        ctx.close()


@gpu
def test_counters_errors_and_switching_off(small_bunny):
    sa, cam = small_bunny
    W, H, N = 64, 48, 8
    rc, rt = scenes.rand_bases(N, 34)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        for err, min_s in ((float("nan"), 16), (-0.1, 16), (0.1, 1)):
            with pytest.raises(capi.FsptError) as e:
                ctx.set_adaptive(err, min_s)
            assert e.value.code == -1
        with pytest.raises(capi.FsptError) as e:
            ctx.read_moment()  # never turned on: there is no moment yet
        assert e.value.code == -3
        ctx.set_adaptive(0.1, 2)
        with pytest.raises(capi.FsptError) as e:
            ctx.render(fr, 0, rc, rt)  # accumulation mode 0
        assert e.value.code == -3
        # every pixel converges at min_samples = 2: later renders add no samples and no rays
        ctx.clear()
        ctx.set_accum_mode(1)
        ctx.set_adaptive(1e30, 2)
        ctx.render(fr, 0, rc[:2], rt[:2])
        acc = ctx.read_accum()
        st = ctx.stats()
        assert (acc[..., 3] == 2).all() and st["samples"] == 2 * W * H and ctx.active_pixels() == 0
        ctx.render(fr, 2, rc[2:], rt[2:])
        st1 = ctx.stats()
        assert st1["samples"] == st["samples"] and st1["rays"] == st["rays"] and st1["last_rays"] == 0
        assert np.array_equal(ctx.read_accum().view(np.uint32), acc.view(np.uint32))
        # off again: the uniform sum-mode render, and the moment is left as it was
        m2 = ctx.read_moment()
        ctx.set_adaptive(0, 2)
        with pytest.raises(capi.FsptError) as e:
            ctx.active_pixels()
        assert e.value.code == -3
        ctx.render(fr, 2, rc[2:], rt[2:])
        assert np.array_equal(ctx.read_moment().view(np.uint32), m2.view(np.uint32))
        ctx.clear()
        ctx.render(fr, 0, rc, rt)
        got = ctx.read_accum()
        assert ctx.stats()["samples"] == N * W * H
    finally:
        ctx.close()
    ref = capi.Context(W, H)
    try:
        ref.scene_upload(sa)
        ref.set_accum_mode(1)
        ref.render(_frame(ref, cam), 0, rc, rt)
        assert np.array_equal(got.view(np.uint32), ref.read_accum().view(np.uint32))
    finally:
        ref.close()


@gpu
def test_converge_stops_when_no_pixel_is_active(small_bunny):
    from fspt_b200.path_tracer import PathTracer
    sa, cam = small_bunny
    pt = PathTracer(sa, (64, 48), cam, max_samples=63)
    try:
        img = pt.converge(0.05, min_samples=8, batch=8)
        n = pt.accumulation()[..., 3]
        assert img.shape == (48, 64, 4) and n.min() >= 8 and n.max() <= 64
        assert pt.pingpong == 64 or pt.ctx.active_pixels() == 0
        assert pt.stats()["samples"] == int(n.sum())
        pt.converge(1e30, min_samples=4, batch=4)  # every pixel stops at 4: the loop ends after its first call
        assert pt.pingpong == 4 and (pt.accumulation()[..., 3] == 4).all()
    finally:
        pt.close()


def test_napi_shim_exposes_the_adaptive_entry_points():
    text = open(os.path.join(ROOT, "fspt_b200", "napi", "fspt_napi.cc")).read()
    for c_name in ("fspt_set_adaptive", "fspt_active_pixels", "fspt_read_moment", "fspt_write_moment"):
        assert re.search(r"\b%s\(" % c_name, text), c_name
    for js_name in ("setAdaptive", "activePixels", "readMoment", "writeMoment"):
        assert '{"%s", ' % js_name in text, js_name
