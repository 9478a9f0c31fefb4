"""fluc_ttmlblend_overlay_set_render_rectangles: gst_video_overlay_rectangle_set_render_rectangle for
the position and size of the composition form's rectangles, scaled again on the GPU from their
resident pixels without a new upload. Every frame is compared at tolerance 0 with the oracle's
composition blend of the rectangle list at the new render rectangles (with the library's model of
the 2x2 chroma mean under averaged chroma).

1. parity on every prepare path (17 formats): grow, shrink, 1x1, 1xN and Nx1, odd sizes and
   origins, across each frame edge, wholly off the frame and back in; a rectangle installed
   unscaled goes scaled and back to its pixel size, one installed scaled goes to other sizes and to
   its pixel size; byte-identical to a fresh overlay_set_rectangles with the same render rectangles
   on another stream; out of place everywhere, and on some steps in place, pinned host frames (zero
   copy) and pageable host frames (staged);
2. the scaler's extremes: a 2x2 source and a 32768x2 source resized;
3. crop: a rectangle with transparent rows and columns whose crop changes with its size;
   lazy_launches and opaque_skip_launches move as for a fresh install of the same list;
4. more resized rectangles than the kernel parameters hold (the uploaded item table);
5. ordering: queued frames keep the old size; one 32-frame batch with every frame at its own size,
   as multi-layout launches and (child process, FLUC_TTMLBLEND_MULTI=0) as table launches;
   submit_many_after followed by a resize;
6. interplay: resize then fade and fade then resize (also installed below 1.0), resize then move
   and move then resize, averaged chroma at every origin parity;
7. cost counters: a size change costs one scale-and-scan launch plus one prepare launch per prepared
   format (plus one per resized rectangle under averaged chroma); a position-only call costs what
   overlay_set_positions costs; an unchanged list costs nothing; h2d_bytes never moves;
8. error codes, each leaving counters and frames as they were;
9. 500 resizes with frames in flight: cache_bytes back at its base after a clear."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from helpers import (PLANAR_420, assert_planes_equal, copy_planes, model_blend, oracle_blend, pkg, random_frame,
                     random_overlay)

pytestmark = pytest.mark.gpu

tbm = pkg.ttmlblend
W, H = 200, 120
FORMATS = ["I420", "YV12", "NV12", "NV21", "Y42B", "Y444", "NV16", "NV24", "YUY2", "UYVY", "GRAY8", "v308",
           "RGB", "AYUV", "RGBA", "BGRA", "ARGB"]
COUNTERS = ("prepare_launches", "h2d_bytes", "overlays_set", "overlays_updated", "cache_bytes")


def cue(seed, ga=1.0):
    """A premultiplied rectangle installed at its pixel size and a straight one installed scaled."""
    return [dict(pixels=random_overlay(60, 40, seed), x=16, y=8, global_alpha=ga),
            dict(pixels=random_overlay(40, 30, seed + 1, premultiplied=False), x=100, y=50, premultiplied=False,
                 global_alpha=ga, render_width=64, render_height=48)]


def sized(rl, rects):
    """rl at the render rectangles (x, y, w, h); a side of 0 is the pixel size."""
    out = []
    for r, (x, y, w, h) in zip(rl, rects):
        ph, pw = r["pixels"].shape[:2]
        out.append(dict(r, x=int(x), y=int(y), render_width=int(w) or pw, render_height=int(h) or ph))
    return out


def faded(rl, alphas):
    return [dict(r, global_alpha=float(a)) for r, a in zip(rl, alphas)]


def blend(ctx, stream, fmt, frame, mode="out", w=W, h=H):
    """One frame through the stream's current overlay: out of place, in place, a pinned host
    frame (zero copy) or a pageable host frame (staged)."""
    if mode == "staged":
        out = copy_planes(frame)
        ctx.wait(ctx.blend_host(stream, fmt, w, h, out))
        return out
    if mode == "zerocopy":
        p = ctx.acquire(fmt, w, h, on_host=True)
        try:
            for dst, src in zip(p.host_planes(), frame):
                dst[...] = src
            for t in ctx.blend_host_many(tbm.TtmlBlend.Batch([stream], fmt, w, h, [p.c], [p.c])):
                ctx.wait(t)
            return [np.array(x) for x in p.host_planes()]
        finally:
            p.release()
    src = ctx.acquire(fmt, w, h)
    try:
        src.upload(frame)
        if mode == "inplace":
            ctx.wait(ctx.submit(stream, fmt, w, h, src.c, src.c))
            return src.download()
        dst = ctx.acquire(fmt, w, h)
        try:
            ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dst.c))
            return dst.download()
        finally:
            dst.release()
    finally:
        src.release()


def expected(fmt, frame, rl, avg=False, w=W, h=H):
    if avg:
        return model_blend(fmt, w, h, copy_planes(frame), rl, chroma_average=True)
    return oracle_blend(fmt, w, h, copy_planes(frame), rl)


MODES_EVERY = ("out",)
MODES_SOME = ("out", "inplace", "zerocopy", "staged")

# (render rectangle of the first, of the second, frame paths)
RESIZES = [
    ((16, 8, 80, 50), (100, 50, 64, 48), MODES_SOME),       # the unscaled one grows (scaled now)
    ((17, 9, 31, 21), (101, 51, 33, 25), MODES_EVERY),      # both shrink, odd sizes and origins
    ((16, 8, 1, 1), (100, 50, 1, 37), MODES_SOME),          # 1x1 and 1xN
    ((15, 7, 57, 1), (99, 49, 37, 1), MODES_EVERY),         # Nx1
    ((-30, -11, 70, 45), (150, 90, 75, 41), MODES_SOME),    # across the left / top and right / bottom edges
    ((-500, 20, 70, 45), (W + 10, 50, 40, 30), MODES_EVERY),  # wholly off the frame (the second unscaled)
    ((16, 8, 0, 0), (100, 50, 0, 0), MODES_SOME),           # back in, both at their pixel size
    ((15, 9, 61, 39), (99, 49, 64, 48), MODES_EVERY),       # scaled again, the second at its install size
    ((3, 2, 60, 40), (120, 71, 40, 30), MODES_SOME),        # pixel sizes given explicitly, moved
    ((3, 2, 123, 77), (120, 71, 40, 30), MODES_EVERY),      # one grows, the other stays
]


@pytest.mark.parametrize("fmt", FORMATS)
def test_resizes_match_oracle(ctx, fmt):
    frame = random_frame(fmt, W, H, 3)
    rl = cue(7)
    st = 1300 + FORMATS.index(fmt)
    fresh = 1330 + FORMATS.index(fmt)
    ctx.overlay_set_rectangles(st, rl)
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, rl), "installed")
    try:
        ctx.set_host_dma(0)                 # pinned host frames: zero copy
        for a, b, modes in RESIZES:
            h0 = ctx.stats()["h2d_bytes"]
            ctx.overlay_set_render_rectangles(st, [a, b])
            assert ctx.stats()["h2d_bytes"] == h0
            now = sized(rl, [a, b])
            want = expected(fmt, frame, now)
            for mode in modes:
                assert_planes_equal(blend(ctx, st, fmt, frame, mode), want, f"{fmt} {a} {b} {mode}")
            ctx.overlay_set_rectangles(fresh, now)              # a fresh install at the same render rectangles
            assert_planes_equal(blend(ctx, fresh, fmt, frame), want, f"{fmt} {a} {b} fresh install")
    finally:
        ctx.set_host_dma(2)


@pytest.mark.parametrize("fmt", ["NV12", "BGRA"])
def test_scaler_extremes(ctx, fmt):
    """The weights at the scaler's extremes: a 2x2 source (every destination pixel between the same
    four), and a 32768x2 source, the widest the scaler takes, resized in both directions."""
    frame = random_frame(fmt, W, H, 4)
    rl = [dict(pixels=random_overlay(2, 2, 21), x=10, y=10),
          dict(pixels=random_overlay(32768, 2, 22, premultiplied=False), x=-16000, y=60, premultiplied=False,
               render_width=32768, render_height=5)]
    st = 1350 + ["NV12", "BGRA"].index(fmt)
    ctx.overlay_set_rectangles(st, rl)
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, rl), "installed")
    for a, b in (((10, 10, 37, 23), (5, 60, 191, 3)), ((11, 9, 1, 9), (-3, 70, 200, 2)),
                 ((10, 10, 2, 2), (-32600, 80, 0, 0)), ((40, 30, 99, 1), (-16383, 20, 32768, 7)),
                 ((10, 10, 32768, 3), (-100, 100, 301, 17))):
        ctx.overlay_set_render_rectangles(st, [a, b])
        now = sized(rl, [a, b])
        for mode in ("out", "inplace"):
            assert_planes_equal(blend(ctx, st, fmt, frame, mode), expected(fmt, frame, now), f"{a} {b} {mode}")


def holey(seed):
    """60x48 with transparent rows and columns and an opaque block: the crop runs and the lazy /
    opaque-skip figures change with the size."""
    px = random_overlay(60, 48, seed)
    px[:6] = 0
    px[18:30] = 0
    px[:, :9] = 0
    px[:, 47:] = 0
    px[32:46, 12:40] = (40, 80, 120, 255)
    return px


def test_crop_follows_the_size(ctx):
    fmt = "NV12"
    frame = random_frame(fmt, W, H, 5)
    rl = [dict(pixels=holey(31), x=20, y=10), dict(pixels=holey(32), x=110, y=40, render_width=70, render_height=60)]
    ctx.overlay_set_rectangles(1360, rl)
    blend(ctx, 1360, fmt, frame)
    for a, b in (((20, 10, 120, 100), (110, 40, 30, 24)), ((21, 11, 61, 13), (111, 39, 80, 79)),
                 ((20, 10, 0, 0), (110, 40, 0, 0)), ((-20, -30, 91, 140), (150, 7, 41, 130))):
        ctx.overlay_set_render_rectangles(1360, [a, b])
        now = sized(rl, [a, b])
        ctx.overlay_set_rectangles(1361, now)
        want = expected(fmt, frame, now)
        d = {}
        for st in (1360, 1361):
            s0 = ctx.stats()
            assert_planes_equal(blend(ctx, st, fmt, frame, "inplace"), want, f"{st} {a} {b} in place")
            assert_planes_equal(blend(ctx, st, fmt, frame, "out"), want, f"{st} {a} {b} out of place")
            s1 = ctx.stats()
            d[st] = (s1["lazy_launches"] - s0["lazy_launches"], s1["opaque_skip_launches"] - s0["opaque_skip_launches"],
                     s1["launches"] - s0["launches"])
        assert d[1360] == d[1361], (a, b, d)


def test_opaque_figures_come_from_the_scaled_pixels(ctx):
    """A 2x2 source opaque on the left and transparent on the right: every scaled pixel but the first
    column mixes the two, so the scaled rectangle has no opaque 16-pixel group while every source
    pixel under it on the left is opaque. In place and out of place launch as for a fresh install."""
    px = np.zeros((2, 2, 4), dtype=np.uint8)
    px[:, 0] = (30, 60, 90, 255)
    rl = [dict(pixels=px, x=10, y=10)]
    fmt = "NV12"
    frame = random_frame(fmt, W, H, 15)
    ctx.overlay_set_rectangles(1365, rl)
    blend(ctx, 1365, fmt, frame)
    for rect in ((10, 10, 96, 64), (11, 9, 160, 100), (10, 10, 2, 2)):
        ctx.overlay_set_render_rectangles(1365, [rect])
        now = sized(rl, [rect])
        ctx.overlay_set_rectangles(1366, now)
        want = expected(fmt, frame, now)
        d = {}
        for st in (1365, 1366):
            s0 = ctx.stats()
            assert_planes_equal(blend(ctx, st, fmt, frame, "inplace"), want, f"{st} {rect} in place")
            assert_planes_equal(blend(ctx, st, fmt, frame, "out"), want, f"{st} {rect} out of place")
            s1 = ctx.stats()
            d[st] = (s1["lazy_launches"] - s0["lazy_launches"], s1["opaque_skip_launches"] - s0["opaque_skip_launches"])
        assert d[1365] == d[1366], (rect, d)


def test_many_rectangles_take_the_uploaded_table(ctx):
    """More resized rectangles than the kernel parameters hold (40): the scale-and-scan items are
    read from device memory."""
    fmt = "I420"
    frame = random_frame(fmt, W, H, 6)
    rl = [dict(pixels=random_overlay(12, 10, 200 + k), x=(k % 8) * 24, y=(k // 8) * 22) for k in range(40)]
    ctx.overlay_set_rectangles(1370, rl)
    blend(ctx, 1370, fmt, frame)
    rects = [((k % 8) * 24 + 1, (k // 8) * 22 + 2, 12 + k % 9, 10 + k % 7) for k in range(40)]
    p0 = ctx.stats()["prepare_launches"]
    ctx.overlay_set_render_rectangles(1370, rects)
    assert ctx.stats()["prepare_launches"] - p0 == 2                 # the scale-and-scan, one batch prepare
    assert_planes_equal(blend(ctx, 1370, fmt, frame), expected(fmt, frame, sized(rl, rects)))


def test_queued_frames_keep_their_size(ctx):
    fmt = "I420"
    rl = cue(41)
    ctx.overlay_set_rectangles(1380, rl)
    frame = random_frame(fmt, W, H, 7)
    src, d1, d2 = ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H)
    src.upload(frame)
    ctx.wait(ctx.submit(1380, fmt, W, H, src.c, d1.c))
    new = [(16, 8, 90, 61), (100, 50, 30, 20)]
    ctx.set_batch(64, 1_000_000)
    try:
        t1 = ctx.submit(1380, fmt, W, H, src.c, d1.c)
        ctx.overlay_set_render_rectangles(1380, new)
        t2 = ctx.submit(1380, fmt, W, H, src.c, d2.c)
        ctx.flush()
        ctx.wait(t1)
        ctx.wait(t2)
    finally:
        ctx.set_batch(32, 200)
    assert_planes_equal(d1.download(), expected(fmt, frame, rl), "queued before the resize")
    assert_planes_equal(d2.download(), expected(fmt, frame, sized(rl, new)), "after the resize")
    # submit_many_after, then a resize before the caller's stream has let the blend run
    tk = ctx.submit_many_after(tbm.TtmlBlend.Batch([1380], fmt, W, H, [src.c], [d1.c]), 0)
    ctx.overlay_set_render_rectangles(1380, [(16, 8, 0, 0), (100, 50, 64, 48)])
    ctx.wait(tk[0])
    assert_planes_equal(d1.download(), expected(fmt, frame, sized(rl, new)), "submit_many_after before the resize")
    assert_planes_equal(blend(ctx, 1380, fmt, frame), expected(fmt, frame, rl), "after it")
    for f in (src, d1, d2):
        f.release()


def check_zoom_inside_one_batch(ctx, stream, w, h):
    """32 frames of one batch, each with the cue at its own size (a caption that zooms in): every
    frame as the oracle blends its own rectangle list. Returns the counters' difference."""
    fmt, n = "NV12", 32
    rl = [dict(pixels=random_overlay(300, 40, 51), x=w - 400, y=h - 80),
          dict(pixels=random_overlay(120, 36, 52, premultiplied=False), x=20, y=10, premultiplied=False)]
    ctx.overlay_set_rectangles(stream, rl)
    frame = random_frame(fmt, w, h, 8)
    src = ctx.acquire(fmt, w, h)
    dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
    src.upload(frame)
    ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dsts[0].c))
    sizes = [[(w - 400 - k, h - 80 - k, 300 + 3 * k, 40 + k), (20, 10, 120 + k, 36 + (k % 5))] for k in range(1, n + 1)]
    ctx.set_batch(64, 1_000_000)
    try:
        st0 = ctx.stats()
        tickets = []
        for rects, d in zip(sizes, dsts):
            ctx.overlay_set_render_rectangles(stream, rects)
            tickets.append(ctx.submit(stream, fmt, w, h, src.c, d.c))
        ctx.flush()
        for t in tickets:
            ctx.wait(t)
        st1 = ctx.stats()
    finally:
        ctx.set_batch(32, 200)
    for k, (rects, d) in enumerate(zip(sizes, dsts)):
        assert_planes_equal(d.download(), expected(fmt, frame, sized(rl, rects), w=w, h=h), f"frame {k}")
    for f in [src] + dsts:
        f.release()
    return {k: st1[k] - st0[k] for k in st0}


def test_zoom_inside_one_batch(ctx):
    d = check_zoom_inside_one_batch(ctx, 1390, 1280, 720)
    assert d["prepare_launches"] == 2 * 32             # a scale-and-scan and a batch prepare per resize
    assert d["h2d_bytes"] == 0
    assert d["launches"] <= 2
    if os.environ.get("FLUC_TTMLBLEND_MULTI", "1") != "0" and os.environ.get("FLUC_TTMLBLEND_GROUPS", "1") != "0":
        assert d["multi_launches"] >= 1                # 32 band lists in one multi-layout launch


TABLE_CHECK = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
from test_gpu_resize import check_zoom_inside_one_batch
import helpers
c = helpers.pkg.TtmlBlend(0)
try:
    d = check_zoom_inside_one_batch(c, 1391, 1280, 720)
    assert d["multi_launches"] == 0, d
    assert 1 <= d["launches"] - d["group_launches"] <= 2, d      # table launches
finally:
    c.close()
print("ok")
"""


def test_zoom_inside_one_batch_as_table_launches(monkeypatch):
    monkeypatch.setenv("FLUC_TTMLBLEND_MULTI", "0")
    here = os.path.dirname(os.path.abspath(__file__))
    out = subprocess.run([sys.executable, "-c", TABLE_CHECK, here, os.path.dirname(here)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout + out.stderr


@pytest.mark.parametrize("fmt", ["NV12", "Y444", "RGB", "BGRA"])
def test_resizes_fades_and_moves(ctx, fmt):
    frame = random_frame(fmt, W, H, 9)
    rl = cue(61)
    st = 1400 + 4 * ["NV12", "Y444", "RGB", "BGRA"].index(fmt)
    ctx.overlay_set_rectangles(st, rl)
    blend(ctx, st, fmt, frame)
    a = [(21, 11, 70, 33), (90, 41, 50, 50)]
    ctx.overlay_set_render_rectangles(st, a)                           # a resize, then a fade
    ctx.overlay_set_global_alpha(st, [0.5, 0.8])
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, faded(sized(rl, a), [0.5, 0.8])),
                        "resize then fade")
    b = [(30, 20, 0, 0), (71, 33, 81, 17)]
    ctx.overlay_set_render_rectangles(st, b)                           # a fade, then a resize
    assert_planes_equal(blend(ctx, st, fmt, frame, "inplace"), expected(fmt, frame, faded(sized(rl, b), [0.5, 0.8])),
                        "fade then resize")
    ctx.overlay_set_positions(st, [5, 60], [3, 70])                    # a resize, then a move: the sizes stay
    c = [(5, 3, 0, 0), (60, 70, 81, 17)]
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, faded(sized(rl, c), [0.5, 0.8])),
                        "resize then move")
    d = [(5, 3, 45, 45), (61, 71, 81, 17)]                             # a move, then a resize
    ctx.overlay_set_render_rectangles(st, d)
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, faded(sized(rl, d), [0.5, 0.8])),
                        "move then resize")
    ctx.overlay_set_rectangles(st, rl)                                 # a new cue starts from its own values
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, rl), "reinstalled")

    low_st = st + 1                                                    # installed at 0.4, then resized
    low = cue(63, ga=0.4)
    ctx.overlay_set_rectangles(low_st, low)
    blend(ctx, low_st, fmt, frame)
    e = [(3, 1, 77, 51), (121, 70, 0, 0)]
    ctx.overlay_set_render_rectangles(low_st, e)
    assert_planes_equal(blend(ctx, low_st, fmt, frame), expected(fmt, frame, sized(low, e)), "0.4 resized")
    ctx.overlay_set_global_alpha(low_st, [0.7, 0.2])
    assert_planes_equal(blend(ctx, low_st, fmt, frame), expected(fmt, frame, faded(sized(low, e), [0.7, 0.2])),
                        "0.4 resized, faded")
    f = [(4, 2, 60, 40), (120, 71, 17, 33)]
    ctx.overlay_set_render_rectangles(low_st, f)
    assert_planes_equal(blend(ctx, low_st, fmt, frame, "inplace"),
                        expected(fmt, frame, faded(sized(low, f), [0.7, 0.2])), "faded, resized")


@pytest.fixture
def averaging(ctx):
    ctx.set_chroma_mode(True)
    try:
        yield ctx
    finally:
        ctx.set_chroma_mode(False)


@pytest.mark.parametrize("fmt", PLANAR_420)
def test_resizes_under_chroma_averaging(averaging, fmt):
    """The averaged chroma of every resized rectangle is prepared at its current global alpha; each
    origin parity puts the 2x2 chroma blocks differently across the rectangle's edges."""
    ctx = averaging
    frame = random_frame(fmt, W, H, 10)
    rl = cue(81)
    st = 1440 + PLANAR_420.index(fmt)
    ctx.overlay_set_rectangles(st, rl)
    blend(ctx, st, fmt, frame)
    ctx.overlay_set_global_alpha(st, [0.6, 1.0])
    k = 0
    for px in (0, 1):
        for py in (0, 1):
            k += 1
            rects = [(20 + px, 10 + py, 61 + k, 37 + px), (101 + py, 51 + px, 45 + py, 29 + k)]
            p0 = ctx.stats()["prepare_launches"]
            ctx.overlay_set_render_rectangles(st, rects)
            # the scale-and-scan, the batch, and each resized rectangle's averaged chroma
            assert ctx.stats()["prepare_launches"] - p0 == 1 + 1 + 2
            want = expected(fmt, frame, faded(sized(rl, rects), [0.6, 1.0]), avg=True)
            for mode in ("out", "inplace"):
                assert_planes_equal(blend(ctx, st, fmt, frame, mode), want, f"{rects} {mode}")


def test_cost_counters(ctx):
    rl = cue(91)
    ctx.overlay_set_rectangles(1450, rl)
    ctx.overlay_set_rectangles(1451, rl)
    frames = {fmt: random_frame(fmt, W, H, 11) for fmt in ("NV12", "RGB", "BGRA")}
    for fmt, f in frames.items():
        blend(ctx, 1450, fmt, f)                       # three prepared formats
        blend(ctx, 1451, fmt, f)
    cur = [(16, 8, 0, 0), (100, 50, 64, 48)]
    for k, new in enumerate(([(16, 8, 81, 50), (100, 50, 64, 48)],      # one resized
                             [(10, 4, 33, 20), (90, 40, 0, 0)],          # both resized and moved
                             [(12, 6, 33, 20), (90, 40, 0, 0)],          # the first only moved
                             [(12, 6, 33, 20), (93, 41, 40, 30)])):      # the second only moved
        st0 = ctx.stats()
        ctx.overlay_set_render_rectangles(1450, new)
        st1 = ctx.stats()
        assert st1["h2d_bytes"] == st0["h2d_bytes"]
        assert st1["overlays_set"] == st0["overlays_set"]
        resized = any((r["render_width"], r["render_height"]) != (q["render_width"], q["render_height"])
                      for r, q in zip(sized(rl, new), sized(rl, cur)))
        if resized:
            assert st1["prepare_launches"] - st0["prepare_launches"] == 1 + 3, new
        else:
            # what overlay_set_positions costs for the same move
            ctx.overlay_set_positions(1451, [n[0] for n in new], [n[1] for n in new])
            st2 = ctx.stats()
            assert st1["prepare_launches"] - st0["prepare_launches"] == 3, new
            assert st2["prepare_launches"] - st1["prepare_launches"] == 3, new
        cur = new
        for fmt, f in frames.items():
            assert_planes_equal(blend(ctx, 1450, fmt, f), expected(fmt, f, sized(rl, new)), f"{fmt} {k}")
    st0 = ctx.stats()
    ctx.overlay_set_render_rectangles(1450, cur)      # unchanged: nothing is done
    ctx.overlay_set_render_rectangles(1450, [(12, 6, 33, 20), (93, 41, 0, 0)])   # 0 = the same pixel size
    st1 = ctx.stats()
    for k in COUNTERS:
        assert st1[k] == st0[k], k


def test_errors(ctx):
    def code(stream, rects):
        with pytest.raises(tbm.TtmlBlendError) as e:
            ctx.overlay_set_render_rectangles(stream, rects)
        return e.value.code

    assert code(1460, [(0, 0, 0, 0)]) == tbm.ERROR_NOT_FOUND          # no overlay yet
    rl = [dict(pixels=random_overlay(60, 40, 95), x=16, y=8),
          dict(pixels=random_overlay(1, 30, 96), x=100, y=50),                        # 1 wide: never scaled
          dict(pixels=random_overlay(40, 30, 97), x=150, y=60, render_width=20, render_height=10)]
    ctx.overlay_set_rectangles(1460, rl)
    fmt = "NV12"
    frame = random_frame(fmt, W, H, 13)
    want = expected(fmt, frame, rl)
    assert_planes_equal(blend(ctx, 1460, fmt, frame), want, "installed")
    now = [(16, 8, 0, 0), (100, 50, 0, 0), (150, 60, 20, 10)]
    big = 2 ** 31 - 1
    bad = [now[:2], now + [(0, 0, 0, 0)],                                       # wrong n
           [(16, 8, -1, 0), now[1], now[2]], [(16, 8, 0, -5), now[1], now[2]],  # negative sides
           [(16, 8, 32769, 0), now[1], now[2]], [now[0], now[1], (150, 60, 5, 32769)],   # above 32768
           [now[0], (100, 50, 2, 30), now[2]], [now[0], (100, 50, 1, 31), now[2]],       # 1x30 would be scaled
           [(big - 59, 8, 0, 0), now[1], now[2]], [(big - 60, 8, 61, 0), now[1], now[2]],  # x + w overflows
           [now[0], now[1], (150, big - 9, 20, 10)], [now[0], now[1], (150, big - 40, 0, 41)]]   # y + h overflows
    st0 = ctx.stats()
    for rects in bad:
        assert code(1460, rects) == tbm.ERROR_INVALID_ARGUMENT, rects
    assert ctx.lib.fluc_ttmlblend_overlay_set_render_rectangles(ctx.h, 1460, None, 3) == tbm.ERROR_INVALID_ARGUMENT
    st1 = ctx.stats()
    for k in COUNTERS:
        assert st1[k] == st0[k], k
    assert_planes_equal(blend(ctx, 1460, fmt, frame), want, "after the refused calls")
    # the last valid ones, and the limits of the scaler
    ctx.overlay_set_render_rectangles(1460, [(big - 60, 8, 0, 0), (100, big - 30, 0, 0), (150, 60, 32768, 1)])
    ctx.overlay_set_render_rectangles(1460, now)
    assert_planes_equal(blend(ctx, 1460, fmt, frame), want, "back")
    # forms that overlay_set_render_rectangles does not resize
    img = random_overlay(W, H, 98)
    ctx.overlay_set(1461, img, [(10, 10, 50, 20)])
    assert code(1461, [(10, 10, 50, 20)]) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_update(1461, img, [(10, 10, 5, 5)])
    assert code(1461, [(10, 10, 50, 20)]) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_set_regions(1462, W, H, [dict(x=10, y=10, w=50, h=20, background_color=0x102030ff)])
    assert code(1462, [(0, 0, 0, 0)]) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_clear(1460)
    assert code(1460, now) == tbm.ERROR_NOT_FOUND
    ctx.overlay_set_rectangles(1463, [])                                # an empty list: n == 0
    ctx.overlay_set_render_rectangles(1463, [])
    assert code(1463, [(0, 0, 0, 0)]) == tbm.ERROR_INVALID_ARGUMENT


def test_resizes_do_not_leak():
    """500 resizes with frames in flight: every generation's scaled blocks, prepared planes and
    tables go back to the pool once no frame holds them; the resident sources with the overlay."""
    c = pkg.TtmlBlend(0)
    try:
        fmt = "NV12"
        frame = random_frame(fmt, W, H, 14)
        src, dst = c.acquire(fmt, W, H), c.acquire(fmt, W, H)
        src.upload(frame)
        c.sync()
        base = c.stats()["cache_bytes"]
        rl = cue(101)
        c.overlay_set_rectangles(1470, rl)
        c.wait(c.submit(1470, fmt, W, H, src.c, dst.c))
        for k in range(500):
            rects = [(16 + k % 37, 8 + k % 5, 40 + k % 41, 30 + k % 23), (100 - k % 29, 50 - k % 7, k % 3 * 32, 0)]
            c.overlay_set_render_rectangles(1470, rects)
            c.submit(1470, fmt, W, H, src.c, dst.c)
        c.sync()
        assert_planes_equal(dst.download(), expected(fmt, frame, sized(rl, rects)), "last resize")
        assert c.stats()["cache_bytes"] > base
        c.overlay_clear(1470)
        c.sync()
        c.sync()        # deferred frees run on the reaper stream after the fences
        deadline = time.time() + 5
        while c.stats()["cache_bytes"] > base and time.time() < deadline:
            time.sleep(0.01)
        assert c.stats()["cache_bytes"] == base
        src.release()
        dst.release()
    finally:
        c.close()
