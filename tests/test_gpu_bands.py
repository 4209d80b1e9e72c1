"""A wave of at least 2 x 2^18 paths is rendered as two row bands on two streams (fspt_api.cu render_wave).  Each
case renders a rectangle large enough to split and compares it bit for bit with the same pixels rendered as row strips
of fewer than 2^19 paths, which render as one band each, and whose equality with the whole frame and with the oracle
test_gpu_api.py::test_tiles_rendered_one_after_the_other_equal_the_whole_frame holds.  Every result is read through the
normal calls, which synchronise only the context's stream: a second stream that was not joined back would leave pixels
unfinished here."""
import numpy as np
import pytest

from fspt_b200 import capi, scenes

pytestmark = pytest.mark.gpu

STATS = ("last_rays", "last_node_visits", "last_leaf_visits")


def _frame(ctx, cam):
    return ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])


def _render(ctx, fr, rect, rc, rt, strip_rows=None):
    """Renders rect (one call, or strips of strip_rows rows); returns the accumulator and the summed counters."""
    ctx.clear()
    x, y, w, h = rect
    strips = [(x, y, w, h)] if strip_rows is None else \
        [(x, y0, w, min(strip_rows, y + h - y0)) for y0 in range(y, y + h, strip_rows)]
    tot = dict.fromkeys(STATS + ("capped_paths",), 0)
    for s in strips:
        before = ctx.stats()["capped_paths"]
        ctx.set_tile(*s)
        ctx.render(fr, 0, rc, rt)
        st = ctx.stats()
        for k in STATS:
            tot[k] += st[k]
        tot["capped_paths"] += st["capped_paths"] - before
    return ctx.read_accum(), tot


def _check(ctx, fr, rect, rc, rt, strip_rows):
    whole, st = _render(ctx, fr, rect, rc, rt)
    strips, st1 = _render(ctx, fr, rect, rc, rt, strip_rows)
    assert np.array_equal(whole.view(np.uint32), strips.view(np.uint32)), rect
    assert st == st1, (rect, st, st1)
    x, y, w, h = rect
    assert float(whole[y:y + h, x:x + w, :3].max()) > 0.0
    return st


def test_frame_split_into_two_tiled_bands(small_bunny):
    """256 x 256 at 32 spp: 2^21 paths, two tiled bands of 128 rows."""
    sa, cam = small_bunny
    rc, rt = scenes.rand_bases(32, 21)
    ctx = capi.Context(256, 256)
    try:
        ctx.scene_upload(sa)
        _check(ctx, _frame(ctx, cam), (0, 0, 256, 256), rc, rt, 16)
    finally:
        ctx.close()


def test_rectangle_with_rows_not_a_multiple_of_8(small_bunny):
    """250 rows: a tiled first band of 124 rows and a row-major second band of 126, both in a sub-rectangle."""
    sa, cam = small_bunny
    rc, rt = scenes.rand_bases(48, 22)
    ctx = capi.Context(272, 260)
    try:
        ctx.scene_upload(sa)
        _check(ctx, _frame(ctx, cam), (8, 3, 256, 250), rc, rt, 20)
    finally:
        ctx.close()


def test_rectangle_too_small_to_split(small_bunny, oracle_mod):
    """Fewer than 4 rows in the first half, or too few paths: one band, still equal to the oracle."""
    sa, cam = small_bunny
    W, H, N = 64, 48, 3
    rc, rt = scenes.rand_bases(N, 23)
    ctx = capi.Context(W, H)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        ctx.clear()
        for rect in [(0, 0, W, 7), (0, 7, W, 41)]:
            ctx.set_tile(*rect)
            ctx.render(fr, 0, rc, rt)
        got = ctx.read_accum()
    finally:
        ctx.close()
    O = oracle_mod.Oracle(sa)
    fb = None
    for k in range(N):
        pos, d = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        fb, _ = O.trace(pos, d, W, H, k, rt[k], cam["env_theta"], fb_prev=fb)
    assert np.array_equal(got[..., :3].view(np.uint32), fb[..., :3].view(np.uint32))


def test_refractive_bands_stop_on_their_own():
    """A refractive prop: each band polls its own path count and stops after its own number of extra bounces; with a
    refraction cap of 1 the capped paths of the two bands differ and their sum is the one-band sum."""
    sa, cam = scenes.pbr_scene(atlas_res=64, subdiv=2, env_size=(128, 64))
    rc, rt = scenes.rand_bases(32, 24)
    ctx = capi.Context(256, 256)
    try:
        ctx.scene_upload(sa)
        fr = _frame(ctx, cam)
        for cap in (64, 1):
            ctx.set_param(capi.PARAM_MAX_REFRACTIONS, cap)
            st = _check(ctx, fr, (0, 0, 256, 256), rc, rt, 16)
            if cap == 1:
                _, top = _render(ctx, fr, (0, 0, 256, 128), rc, rt, 16)
                _, bottom = _render(ctx, fr, (0, 128, 256, 128), rc, rt, 16)
                assert top["capped_paths"] + bottom["capped_paths"] == st["capped_paths"] > 0
                assert top["capped_paths"] != bottom["capped_paths"], (top, bottom)
    finally:
        ctx.close()


def test_render_longer_than_one_wave(small_bunny, monkeypatch):
    """3 samples per wave, 7 samples: two split waves of 3 and a last wave of 1 sample too small to split.  That last
    wave renders both bands' rows on the context's stream; it is ordered behind the second stream's last band because
    fspt_render makes the two streams wait for each other before a wave of another size."""
    monkeypatch.setenv("FSPT_WAVE_SAMPLES", "3")
    sa, cam = small_bunny
    rc, rt = scenes.rand_bases(7, 25)
    ctx = capi.Context(512, 384)
    try:
        ctx.scene_upload(sa)
        _check(ctx, _frame(ctx, cam), (0, 0, 512, 384), rc, rt, 32)
    finally:
        ctx.close()


def test_sum_mode_tile(small_bunny):
    """Sum mode (per-pixel sample count in alpha) in a tile of the frame."""
    sa, cam = small_bunny
    rc, rt = scenes.rand_bases(40, 26)
    ctx = capi.Context(320, 288)
    try:
        ctx.scene_upload(sa)
        ctx.set_accum_mode(1)
        fr = _frame(ctx, cam)
        _check(ctx, fr, (16, 24, 256, 224), rc, rt, 16)
        acc = ctx.read_accum()
        assert (acc[24:248, 16:272, 3] == 40.0).all() and (acc[:24, :, 3] == 0.0).all()
    finally:
        ctx.close()


def test_last_wave_split_with_fewer_samples(small_bunny, monkeypatch):
    """4 samples per wave, 7 samples: the last wave of 3 samples is still split (3 x 512 x 192 >= 2^18 paths per band),
    with other slice offsets than the first wave's bands."""
    monkeypatch.setenv("FSPT_WAVE_SAMPLES", "4")
    sa, cam = small_bunny
    rc, rt = scenes.rand_bases(7, 27)
    ctx = capi.Context(512, 384)
    try:
        ctx.scene_upload(sa)
        _check(ctx, _frame(ctx, cam), (0, 0, 512, 384), rc, rt, 32)
    finally:
        ctx.close()
