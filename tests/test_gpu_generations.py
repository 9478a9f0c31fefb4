"""A new generation of a stream's overlay (overlay_update, overlay_set_global_alpha,
overlay_set_positions) keeps the prepared planes of every rectangle that did not change for the
prepare, and prepares only the others. The frames would come out exact either way, so these tests
count prepare launches, and check each frame against the oracle besides.

1. update: touching one of three region boxes prepares what installing that box alone does;
2. move under averaged chroma: moving one of two rectangles is the batch plus its averaged chroma;
3. fade: fading one of two PLANE8 rectangles installed at 0.4 prepares that rectangle only."""
import numpy as np
import pytest

from helpers import assert_planes_equal, copy_planes, model_blend, oracle_blend, random_frame, random_overlay, wl
from oracle import oracle

pytestmark = pytest.mark.gpu

W, H = 320, 180
REGIONS = [wl.Region(16, 8, 280, 40, (0, 0, 0, 255), 0.8),
           wl.Region(24, 70, 150, 40, (0, 0, 128, 255), 0.5, ((255, 255, 0, 255),)),
           wl.Region(40, 130, 240, 40, (32, 32, 32, 255), 1.0)]
BOXES = [(r.x, r.y, r.w, r.h) for r in REGIONS]


def region_image(seeds):
    img = np.zeros((H, W, 4), dtype=np.uint8)
    for k, (reg, seed) in enumerate(zip(REGIONS, seeds)):
        one = wl.make_overlay(W, H, [reg], 6000 + 10 * seed + k)
        img[reg.y:reg.y + reg.h, reg.x:reg.x + reg.w] = one[reg.y:reg.y + reg.h, reg.x:reg.x + reg.w]
    return img


def blend(ctx, stream, fmt, frame):
    src, dst = ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H)
    try:
        src.upload(frame)
        ctx.wait(ctx.submit(stream, fmt, W, H, src.c, dst.c))
        return dst.download()
    finally:
        src.release()
        dst.release()


def launches(ctx):
    return ctx.stats()["prepare_launches"]


def two_rects(seed, ga=1.0):
    return [dict(pixels=random_overlay(60, 40, seed), x=17, y=9, global_alpha=ga),
            dict(pixels=random_overlay(64, 48, seed + 1, premultiplied=False), x=151, y=71, premultiplied=False,
                 global_alpha=ga)]


def test_update_prepares_only_the_touched_box(ctx):
    fmt = "NV12"
    frame = random_frame(fmt, W, H, 1)
    a, b = region_image([1, 1, 1]), region_image([1, 2, 1])
    ctx.overlay_set(1300, a, BOXES)
    blend(ctx, 1300, fmt, frame)                        # prepared for NV12: the update prepares for it at once
    p0 = launches(ctx)
    ctx.overlay_update(1300, b, [BOXES[1]])
    update = launches(ctx) - p0
    want = oracle_blend(fmt, W, H, copy_planes(frame), oracle.ttmlrender_rectangles(b))
    assert_planes_equal(blend(ctx, 1300, fmt, frame), want, "after the update")

    p0 = launches(ctx)
    ctx.overlay_set(1301, b, [BOXES[1]])                # the touched box alone, on a stream of its own
    blend(ctx, 1301, fmt, frame)
    alone = launches(ctx) - p0
    assert alone > 0
    assert update == alone


def test_move_of_one_rectangle_under_chroma_averaging(ctx):
    fmt = "I420"
    frame = random_frame(fmt, W, H, 2)
    rl = two_rects(20)
    ctx.set_chroma_mode(True)
    try:
        ctx.overlay_set_rectangles(1302, rl)
        blend(ctx, 1302, fmt, frame)
        p0 = launches(ctx)
        ctx.overlay_set_positions(1302, [17, 160], [9, 74])        # only the second one moves
        assert launches(ctx) - p0 == 1 + 1      # the batch, plus the moved rectangle's averaged chroma
        moved = [rl[0], dict(rl[1], x=160, y=74)]
        want = model_blend(fmt, W, H, copy_planes(frame), moved, chroma_average=True)
        assert_planes_equal(blend(ctx, 1302, fmt, frame), want, "after the move")
    finally:
        ctx.set_chroma_mode(False)


def test_fade_of_one_plane8_rectangle_installed_below_one(ctx):
    fmt = "NV12"
    frame = random_frame(fmt, W, H, 3)
    rl = two_rects(30, ga=0.4)
    ctx.overlay_set_rectangles(1303, rl)
    blend(ctx, 1303, fmt, frame)
    p0 = launches(ctx)
    ctx.overlay_set_global_alpha(1303, [0.4, 0.8])               # only the second one changes
    fade = launches(ctx) - p0
    want = oracle_blend(fmt, W, H, copy_planes(frame), [rl[0], dict(rl[1], global_alpha=0.8)])
    assert_planes_equal(blend(ctx, 1303, fmt, frame), want, "after the fade")

    p0 = launches(ctx)
    ctx.overlay_set_rectangles(1304, [rl[1]])           # that rectangle alone, on a stream of its own
    blend(ctx, 1304, fmt, frame)
    alone = launches(ctx) - p0
    assert alone > 0
    assert fade == alone
