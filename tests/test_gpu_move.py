"""fluc_ttmlblend_overlay_set_positions: gst_video_overlay_rectangle_set_render_rectangle for the
position of the composition form's rectangles, without a new upload, scale or scan. Every frame is
compared with the oracle's composition blend of the moved rectangle list at tolerance 0.

1. parity on every prepare path (17 formats): every dx in 0..33 and dy in 0..3 (both parities, the
   4-, 16- and 32-pixel grid periods), across each frame edge, wholly off the frame and back in;
   byte-identical to a fresh overlay_set_rectangles at the same positions on another stream; out of
   place, in place, pinned host frames (zero copy) and pageable host frames (staged);
2. rectangles installed at negative x / y, or wholly above / left of the frame, moved in;
3. ordering: queued frames keep the old position; one 32-frame batch with every frame at its own
   position, as multi-layout launches and (child process, FLUC_TTMLBLEND_MULTI=0) as table
   launches; submit_many_after followed by a move;
4. interplay with global alpha (move then fade, fade then move, installed below 1.0), a scaled
   rectangle, and averaged chroma at every origin parity;
5. cost counters: no h2d bytes, one prepare launch per prepared format;
6. error codes and unchanged positions;
7. 500 moves with frames in flight: cache_bytes back at its base."""
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


def cue(seed, ga=1.0):
    """A premultiplied and a straight rectangle that overlap after some moves."""
    return [dict(pixels=random_overlay(60, 40, seed), x=16, y=8, global_alpha=ga),
            dict(pixels=random_overlay(64, 48, seed + 1, premultiplied=False), x=100, y=50, premultiplied=False,
                 global_alpha=ga)]


def at(rl, xs, ys):
    return [dict(r, x=int(x), y=int(y)) for r, x, y in zip(rl, xs, ys)]


def faded(rl, alphas):
    if np.ndim(alphas) == 0:
        alphas = [alphas] * len(rl)
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


def moves():
    """(xs, ys, modes): every dx in 0..33 and dy in 0..3, then across the edges, off and back in."""
    out = []
    for dy in range(4):
        for dx in range(34):
            modes = MODES_SOME if dx in (1, 16, 33) and dy in (0, 3) else MODES_EVERY
            out.append(([16 + dx, 100 - dx], [8 + dy, 50 + dy], modes))
    for xs, ys in (([-30, 150], [8, 50]), ([-59, 170], [-39, 100]), ([-7, W - 3], [-3, H - 1]),
                   ([-600, W + 40], [-500, 50]), ([16, 100], [H + 5, -48]), ([W, 100], [8, -47]),
                   ([15, 101], [9, 49])):
        out.append((xs, ys, MODES_SOME))
    return out


@pytest.mark.parametrize("fmt", FORMATS)
def test_moves_match_oracle(ctx, fmt):
    frame = random_frame(fmt, W, H, 3)
    rl = cue(7)
    ctx.overlay_set_rectangles(1100, rl)
    assert_planes_equal(blend(ctx, 1100, fmt, frame), expected(fmt, frame, rl), "before the move")
    try:
        ctx.set_host_dma(0)                 # pinned host frames: zero copy
        for xs, ys, modes in moves():
            ctx.overlay_set_positions(1100, xs, ys)
            moved = at(rl, xs, ys)
            want = expected(fmt, frame, moved)
            for mode in modes:
                assert_planes_equal(blend(ctx, 1100, fmt, frame, mode), want, f"{fmt} {xs} {ys} {mode}")
            ctx.overlay_set_rectangles(1101, moved)             # a fresh install at the same positions
            assert_planes_equal(blend(ctx, 1101, fmt, frame), want, f"{fmt} {xs} {ys} fresh install")
    finally:
        ctx.set_host_dma(2)


@pytest.mark.parametrize("fmt", ["I420", "NV12", "YUY2", "RGB", "BGRA"])
def test_rectangles_off_the_left_and_top_move_in(ctx, fmt):
    frame = random_frame(fmt, W, H, 4)
    rl = [dict(pixels=random_overlay(70, 50, 31), x=-40, y=-21),                # hangs off the top-left corner
          dict(pixels=random_overlay(50, 40, 33, premultiplied=False), x=-200, y=30, premultiplied=False),
          dict(pixels=random_overlay(40, 30, 35), x=60, y=-100)]                 # wholly above
    ctx.overlay_set_rectangles(1110, rl)
    assert_planes_equal(blend(ctx, 1110, fmt, frame), expected(fmt, frame, rl), "installed")
    for xs, ys in (([11, 90, 150], [5, 60, 80]), ([-39, -49, 60], [-20, 30, -29]), ([0, 0, 0], [0, 0, 0])):
        ctx.overlay_set_positions(1110, xs, ys)
        for mode in ("out", "inplace"):
            assert_planes_equal(blend(ctx, 1110, fmt, frame, mode), expected(fmt, frame, at(rl, xs, ys)),
                                f"{xs} {ys} {mode}")


def test_queued_frames_keep_their_position(ctx):
    fmt = "I420"
    rl = cue(41)
    ctx.overlay_set_rectangles(1120, rl)
    frame = random_frame(fmt, W, H, 5)
    src, d1, d2 = ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H)
    src.upload(frame)
    ctx.wait(ctx.submit(1120, fmt, W, H, src.c, d1.c))
    ctx.set_batch(64, 1_000_000)
    try:
        t1 = ctx.submit(1120, fmt, W, H, src.c, d1.c)
        ctx.overlay_set_positions(1120, [17, 99], [9, 51])
        t2 = ctx.submit(1120, fmt, W, H, src.c, d2.c)
        ctx.flush()
        ctx.wait(t1)
        ctx.wait(t2)
    finally:
        ctx.set_batch(32, 200)
    assert_planes_equal(d1.download(), expected(fmt, frame, rl), "queued before the move")
    assert_planes_equal(d2.download(), expected(fmt, frame, at(rl, [17, 99], [9, 51])), "after the move")
    # submit_many_after, then a move before the caller's stream has let the blend run
    ctx.overlay_set_positions(1120, [16, 100], [8, 50])
    tk = ctx.submit_many_after(tbm.TtmlBlend.Batch([1120], fmt, W, H, [src.c], [d1.c]), 0)
    ctx.overlay_set_positions(1120, [40, 20], [30, 70])
    ctx.wait(tk[0])
    assert_planes_equal(d1.download(), expected(fmt, frame, rl), "submit_many_after before the move")
    for f in (src, d1, d2):
        f.release()


def check_scroll_inside_one_batch(ctx, stream, w, h):
    """32 frames of one batch, each at its own position (a ticker): one launch per layout class,
    every frame as the oracle blends its own rectangle list. Returns the counters' difference."""
    fmt, n = "NV12", 32
    rl = [dict(pixels=random_overlay(300, 40, 51), x=w - 300, y=h - 60),
          dict(pixels=random_overlay(120, 36, 52, premultiplied=False), x=20, y=10, premultiplied=False)]
    ctx.overlay_set_rectangles(stream, rl)
    frame = random_frame(fmt, w, h, 6)
    src = ctx.acquire(fmt, w, h)
    dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
    src.upload(frame)
    ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dsts[0].c))
    pos = [([w - 300 - 7 * k, 20 + k], [h - 60 - (k % 4), 10 + k // 2]) for k in range(1, n + 1)]
    ctx.set_batch(64, 1_000_000)
    try:
        st0 = ctx.stats()
        tickets = []
        for (xs, ys), d in zip(pos, dsts):
            ctx.overlay_set_positions(stream, xs, ys)
            tickets.append(ctx.submit(stream, fmt, w, h, src.c, d.c))
        ctx.flush()
        for t in tickets:
            ctx.wait(t)
        st1 = ctx.stats()
    finally:
        ctx.set_batch(32, 200)
    for k, ((xs, ys), d) in enumerate(zip(pos, dsts)):
        assert_planes_equal(d.download(), expected(fmt, frame, at(rl, xs, ys), w=w, h=h), f"frame {k}")
    for f in [src] + dsts:
        f.release()
    return {k: st1[k] - st0[k] for k in st0}


def test_scroll_inside_one_batch(ctx):
    d = check_scroll_inside_one_batch(ctx, 1130, 1280, 720)
    assert d["prepare_launches"] == 32                 # one batch prepare per move (one format)
    assert d["h2d_bytes"] == 0
    assert d["launches"] <= 2
    if os.environ.get("FLUC_TTMLBLEND_MULTI", "1") != "0" and os.environ.get("FLUC_TTMLBLEND_GROUPS", "1") != "0":
        assert d["multi_launches"] >= 1                # 32 band lists in one multi-layout launch


TABLE_CHECK = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
from test_gpu_move import check_scroll_inside_one_batch
import helpers
c = helpers.pkg.TtmlBlend(0)
try:
    d = check_scroll_inside_one_batch(c, 1131, 1280, 720)
    assert d["multi_launches"] == 0, d
    assert 1 <= d["launches"] - d["group_launches"] <= 2, d      # table launches
finally:
    c.close()
print("ok")
"""


def test_scroll_inside_one_batch_as_table_launches(monkeypatch):
    monkeypatch.setenv("FLUC_TTMLBLEND_MULTI", "0")
    here = os.path.dirname(os.path.abspath(__file__))
    out = subprocess.run([sys.executable, "-c", TABLE_CHECK, here, os.path.dirname(here)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout + out.stderr


@pytest.mark.parametrize("fmt", ["NV12", "Y444", "RGB", "BGRA"])
def test_moves_and_fades(ctx, fmt):
    frame = random_frame(fmt, W, H, 8)
    rl = cue(61)
    ctx.overlay_set_rectangles(1140, rl)
    blend(ctx, 1140, fmt, frame)
    ctx.overlay_set_positions(1140, [21, 90], [11, 41])               # a move, then a fade
    ctx.overlay_set_global_alpha(1140, [0.5, 0.8])
    want = expected(fmt, frame, faded(at(rl, [21, 90], [11, 41]), [0.5, 0.8]))
    assert_planes_equal(blend(ctx, 1140, fmt, frame), want, "move then fade")
    ctx.overlay_set_positions(1140, [30, 71], [20, 33])               # a fade, then a move
    want = expected(fmt, frame, faded(at(rl, [30, 71], [20, 33]), [0.5, 0.8]))
    assert_planes_equal(blend(ctx, 1140, fmt, frame, "inplace"), want, "fade then move")
    ctx.overlay_set_rectangles(1140, rl)                               # a new cue starts from its own values
    assert_planes_equal(blend(ctx, 1140, fmt, frame), expected(fmt, frame, rl), "reinstalled")

    st = 1141 + FORMATS.index(fmt)                                     # installed at 0.4, then moved
    low = cue(63, ga=0.4)
    ctx.overlay_set_rectangles(st, low)
    blend(ctx, st, fmt, frame)
    ctx.overlay_set_positions(st, [3, 121], [1, 70])
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, at(low, [3, 121], [1, 70])), "0.4 moved")
    ctx.overlay_set_global_alpha(st, [0.7, 0.2])
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, faded(at(low, [3, 121], [1, 70]),
                                                                               [0.7, 0.2])), "0.4 moved, faded")
    ctx.overlay_set_positions(st, [4, 120], [2, 71])
    assert_planes_equal(blend(ctx, st, fmt, frame, "inplace"),
                        expected(fmt, frame, faded(at(low, [4, 120], [2, 71]), [0.7, 0.2])), "faded, moved")


@pytest.mark.parametrize("fmt", ["NV12", "I420", "RGBA"])
def test_scaled_rectangle_moves_without_an_upload(ctx, fmt):
    frame = random_frame(fmt, W, H, 9)
    rl = [dict(pixels=random_overlay(40, 30, 71), x=10, y=10, render_width=90, render_height=55),
          dict(pixels=random_overlay(30, 20, 72), x=120, y=60)]
    ctx.overlay_set_rectangles(1160, rl)
    blend(ctx, 1160, fmt, frame)
    for xs, ys in (([13, 101], [7, 61]), ([-20, 150], [80, -5]), ([150, 0], [90, 0])):
        h0 = ctx.stats()["h2d_bytes"]
        ctx.overlay_set_positions(1160, xs, ys)
        assert ctx.stats()["h2d_bytes"] == h0
        assert_planes_equal(blend(ctx, 1160, fmt, frame), expected(fmt, frame, at(rl, xs, ys)), f"{xs} {ys}")


@pytest.fixture
def averaging(ctx):
    ctx.set_chroma_mode(True)
    try:
        yield ctx
    finally:
        ctx.set_chroma_mode(False)


@pytest.mark.parametrize("fmt", PLANAR_420)
def test_moves_under_chroma_averaging(averaging, fmt):
    """The averaged chroma of every moved rectangle is prepared again at its current global alpha;
    each origin parity puts the 2x2 chroma blocks differently across the rectangle's edges."""
    ctx = averaging
    frame = random_frame(fmt, W, H, 10)
    rl = cue(81)
    st = 1170 + PLANAR_420.index(fmt)
    ctx.overlay_set_rectangles(st, rl)
    blend(ctx, st, fmt, frame)
    ctx.overlay_set_global_alpha(st, [0.6, 1.0])
    for px in (0, 1):
        for py in (0, 1):
            xs, ys = [20 + px, 101 + py], [10 + py, 51 + px]
            p0 = ctx.stats()["prepare_launches"]
            ctx.overlay_set_positions(st, xs, ys)
            assert ctx.stats()["prepare_launches"] - p0 == 1 + 2      # the batch, plus each averaged chroma
            want = expected(fmt, frame, faded(at(rl, xs, ys), [0.6, 1.0]), avg=True)
            for mode in ("out", "inplace"):
                assert_planes_equal(blend(ctx, st, fmt, frame, mode), want, f"{xs} {ys} {mode}")


def test_cost_counters(ctx):
    rl = cue(91)
    ctx.overlay_set_rectangles(1180, rl)
    frames = {fmt: random_frame(fmt, W, H, 11) for fmt in ("NV12", "RGB", "BGRA")}
    for fmt, f in frames.items():
        blend(ctx, 1180, fmt, f)                       # three prepared formats
    for k, (xs, ys) in enumerate((([17, 99], [9, 49]), ([50, 10], [60, 20]), ([-10, 180], [-5, 100]))):
        st0 = ctx.stats()
        ctx.overlay_set_positions(1180, xs, ys)
        st1 = ctx.stats()
        assert st1["h2d_bytes"] == st0["h2d_bytes"]
        assert st1["prepare_launches"] - st0["prepare_launches"] == 3, (xs, ys)   # one per format, no scale
        assert st1["overlays_set"] == st0["overlays_set"]
        for fmt, f in frames.items():
            assert_planes_equal(blend(ctx, 1180, fmt, f), expected(fmt, f, at(rl, xs, ys)), f"{fmt} {k}")


def test_many_rectangles_take_the_uploaded_batch(ctx):
    """More prepare items than the kernel parameters hold (40 rectangles x 2 planes on I420): the
    batch's items are read from device memory."""
    fmt = "I420"
    frame = random_frame(fmt, W, H, 12)
    rl = [dict(pixels=random_overlay(12, 10, 200 + k), x=(k % 8) * 24, y=(k // 8) * 22) for k in range(40)]
    ctx.overlay_set_rectangles(1190, rl)
    blend(ctx, 1190, fmt, frame)
    xs = [(k % 8) * 24 + 5 for k in range(40)]
    ys = [(k // 8) * 22 + 3 for k in range(40)]
    p0 = ctx.stats()["prepare_launches"]
    ctx.overlay_set_positions(1190, xs, ys)
    assert ctx.stats()["prepare_launches"] - p0 == 1
    assert_planes_equal(blend(ctx, 1190, fmt, frame), expected(fmt, frame, at(rl, xs, ys)))


def test_errors(ctx):
    def code(stream, xs, ys):
        with pytest.raises(tbm.TtmlBlendError) as e:
            ctx.overlay_set_positions(stream, xs, ys)
        return e.value.code

    assert code(1200, [0], [0]) == tbm.ERROR_NOT_FOUND                  # no overlay yet
    rl = cue(95)
    ctx.overlay_set_rectangles(1200, rl)
    assert code(1200, [1], [1]) == tbm.ERROR_INVALID_ARGUMENT           # wrong n
    assert code(1200, [1, 2, 3], [1, 2, 3]) == tbm.ERROR_INVALID_ARGUMENT
    arr = (tbm.C.c_int32 * 2)(1, 2)
    assert ctx.lib.fluc_ttmlblend_overlay_set_positions(ctx.h, 1200, None, arr, 2) == tbm.ERROR_INVALID_ARGUMENT
    assert ctx.lib.fluc_ttmlblend_overlay_set_positions(ctx.h, 1200, arr, None, 2) == tbm.ERROR_INVALID_ARGUMENT
    big = 2 ** 31 - 1
    assert code(1200, [big - 59, 0], [0, 0]) == tbm.ERROR_INVALID_ARGUMENT    # x + 60 overflows
    assert code(1200, [0, 0], [0, big - 47]) == tbm.ERROR_INVALID_ARGUMENT    # y + 48 overflows
    ctx.overlay_set_positions(1200, [big - 60, 0], [0, big - 48])              # the last valid ones
    ctx.overlay_set_positions(1200, [-big - 1, 0], [-big - 1, 0])
    # unchanged positions: nothing is done
    ctx.overlay_set_positions(1200, [16, 100], [8, 50])
    frame = random_frame("NV12", W, H, 13)
    blend(ctx, 1200, "NV12", frame)
    st0 = ctx.stats()
    ctx.overlay_set_positions(1200, [16, 100], [8, 50])
    st1 = ctx.stats()
    assert st1["prepare_launches"] == st0["prepare_launches"]
    assert_planes_equal(blend(ctx, 1200, "NV12", frame), expected("NV12", frame, rl), "unchanged")
    # forms that overlay_set_positions does not move
    img = random_overlay(W, H, 96)
    ctx.overlay_set(1201, img, [(10, 10, 50, 20)])
    assert code(1201, [0], [0]) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_update(1201, img, [(10, 10, 5, 5)])
    assert code(1201, [0], [0]) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_set_regions(1202, W, H, [dict(x=10, y=10, w=50, h=20, background_color=0x102030ff)])
    assert code(1202, [0], [0]) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_clear(1200)
    assert code(1200, [16, 100], [8, 50]) == tbm.ERROR_NOT_FOUND
    ctx.overlay_set_rectangles(1203, [])                                # an empty list: n == 0
    ctx.overlay_set_positions(1203, [], [])
    assert code(1203, [0], [0]) == tbm.ERROR_INVALID_ARGUMENT


def test_moves_do_not_leak():
    """500 moves with frames in flight: every generation's prepared planes and tables go back to
    the pool once no frame holds them."""
    c = pkg.TtmlBlend(0)
    try:
        fmt = "NV12"
        frame = random_frame(fmt, W, H, 14)
        src, dst = c.acquire(fmt, W, H), c.acquire(fmt, W, H)
        src.upload(frame)
        c.sync()
        base = c.stats()["cache_bytes"]
        rl = cue(101)
        c.overlay_set_rectangles(1210, rl)
        c.wait(c.submit(1210, fmt, W, H, src.c, dst.c))
        for k in range(500):
            xs, ys = [16 + k % 37, 100 - k % 29], [8 + k % 5, 50 - k % 7]
            c.overlay_set_positions(1210, xs, ys)
            c.submit(1210, fmt, W, H, src.c, dst.c)
        c.sync()
        assert_planes_equal(dst.download(), expected(fmt, frame, at(rl, xs, ys)), "last move")
        assert c.stats()["cache_bytes"] > base
        c.overlay_clear(1210)
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
