"""fluc_ttmlblend_overlay_set_global_alpha: gst_video_overlay_rectangle_set_global_alpha for the
stream's current overlay, applied per frame without a new upload or prepare. Every frame is
compared with the oracle's composition blend of the same rectangles at the new global alphas,
at tolerance 0.

1. every plane kind (PLANE8, PLANE8_RGB, both packed kinds), alphas 0, 1/255, 0.5, 254/255 and
   1, straight and premultiplied sources and destinations, in and out of place;
2. one value per rectangle on three overlapping rectangles, and the n == 1 form;
3. a fade inside one batch: 32 frames, each with its own value, one launch, no prepare;
4. frames already queued keep the value they were submitted with;
5. lifecycle: overlay_update keeps the value, overlay_set starts again at 1, a cue installed at
   0.4 is prepared once more the first time it is faded and never again;
6. a cue with an opaque box (opaque skip, lazy in place) faded to 0.5, with the lazy and
   opaque-skip knobs forced on and off (in a child process: the library reads them once);
7. host frames: pinned zero copy, host DMA batches, pageable frames through the staging
   threads, and submit_many_after;
8. global alpha 0: out of place the copy, in place nothing is touched and nothing launched;
9. the error codes;
10. the same fades under FLUC_TTMLBLEND_CHROMA_AVERAGE on the four 4:2:0 formats, at odd
   origins, against model_blend(chroma_average=True) at the faded values: per-rectangle values,
   a fade inside one batch, queued frames, overlay_update of a faded box, and the cache's memory
   back at its baseline once the cues are cleared."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import (PLANAR_420, assert_planes_equal, copy_planes, gpu_blend, model_blend, oracle_blend, pkg,
                     random_frame, random_overlay, wl)
from oracle import oracle

pytestmark = pytest.mark.gpu

tbm = pkg.ttmlblend
W, H = 200, 120            # 200: ragged last vectors of some planes -> byte-granular table jobs too
FORMATS = ["NV12", "I420", "Y444", "YUY2", "GRAY8", "v308", "RGB", "BGR", "AYUV", "ARGB", "RGBA", "BGRA"]
ALPHAS = [0.0, 1 / 255, 0.5, 254 / 255, 1.0]


def rects(seed, sp=True, ga=1.0, w=W):
    """Two overlapping rectangles: one-rectangle windows and general windows."""
    return [dict(pixels=random_overlay(120, 50, seed, premultiplied=sp), x=16, y=8, global_alpha=ga,
                 premultiplied=sp),
            dict(pixels=random_overlay(64, 80, seed + 1, premultiplied=sp), x=w - 100, y=30,
                 global_alpha=ga, premultiplied=sp)]


def faded(rl, alphas):
    if np.ndim(alphas) == 0:
        alphas = [alphas] * len(rl)
    return [dict(r, global_alpha=float(a)) for r, a in zip(rl, alphas)]


def blend(ctx, stream, fmt, frame, mode="out", dp=False, w=W, h=H):
    return gpu_blend(ctx, fmt, w, h, frame, mode=mode, stream=stream, dest_premul=dp, set_overlay=False)


def expected(fmt, frame, rl, dp=False, avg=False, w=W, h=H):
    """The oracle's blend; under chroma averaging the numpy model of that option (its luma is the
    oracle's, which is checked too)."""
    want = oracle_blend(fmt, w, h, copy_planes(frame), rl, dp)
    if not avg:
        return want
    got = model_blend(fmt, w, h, copy_planes(frame), rl, dp, chroma_average=True)
    assert np.array_equal(got[0], want[0])
    return got


@pytest.fixture
def averaging(ctx):
    """The session context with FLUC_TTMLBLEND_CHROMA_AVERAGE for one test."""
    ctx.set_chroma_mode(True)
    try:
        yield ctx
    finally:
        ctx.set_chroma_mode(False)


def odd_rects(seed, sp=True, ga=1.0, w=W):
    """rects() at odd origins: 2x2 chroma blocks half inside, half outside every rectangle."""
    return [dict(r, x=r["x"] + 1, y=r["y"] + 1) for r in rects(seed, sp, ga, w)]


def check_faded_cue(ctx, fmt, alpha, avg=False):
    frame = random_frame(fmt, W, H, 7)
    for sp in (True, False):
        rl = (odd_rects if avg else rects)(11, sp)
        ctx.overlay_set_rectangles(900, rl)
        # one frame at 1.0 first, so that the fade re-uses prepared planes instead of preparing them
        assert_planes_equal(blend(ctx, 900, fmt, frame), expected(fmt, frame, rl, avg=avg), f"{fmt} before the fade")
        ctx.overlay_set_global_alpha(900, alpha)
        for dp in (False, True):
            want = expected(fmt, frame, faded(rl, alpha), dp, avg)
            for mode in ("out", "inplace"):
                assert_planes_equal(blend(ctx, 900, fmt, frame, mode, dp), want,
                                    f"{fmt} ga={alpha} sp={sp} dp={dp} {mode}")


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("fmt", FORMATS)
def test_faded_cue_matches_oracle(ctx, fmt, alpha):
    check_faded_cue(ctx, fmt, alpha)


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("fmt", PLANAR_420)
def test_faded_cue_under_chroma_averaging(averaging, fmt, alpha):
    """The averaged chroma sample weighs its four pixels by asrc = a*ga/255 (BLENDSPEC section 7),
    so a fade gives what installing the rectangles at the new value gives."""
    check_faded_cue(averaging, fmt, alpha, avg=True)


@pytest.mark.parametrize("fmt", ["NV12", "Y444", "RGB", "BGRA"])
def test_fade_before_the_first_frame(ctx, fmt):
    """A fade of a cue no frame has used yet: the first frame prepares it, without a global alpha."""
    frame = random_frame(fmt, W, H, 8)
    rl = rects(13)
    ctx.overlay_set_rectangles(906, rl)
    ctx.overlay_set_global_alpha(906, 0.3)
    assert_planes_equal(blend(ctx, 906, fmt, frame), oracle_blend(fmt, W, H, copy_planes(frame), faded(rl, 0.3)))


def check_per_rectangle_values(ctx, fmt, avg=False):
    frame = random_frame(fmt, W, H, 9)
    o = 1 if avg else 0
    rl = [dict(pixels=random_overlay(90, 60, 21), x=10 + o, y=10 + o),
          dict(pixels=random_overlay(90, 60, 22, premultiplied=False), x=50 + o, y=30 + o, premultiplied=False),
          dict(pixels=random_overlay(90, 60, 23), x=80 + o, y=50 + o)]
    ctx.overlay_set_rectangles(910, rl)
    blend(ctx, 910, fmt, frame)
    for alphas in ([0.3, 0.0, 0.9], [1.0, 0.6, 0.25], [0.75], [0.75, 0.5, 0.75]):
        ctx.overlay_set_global_alpha(910, alphas)
        want = expected(fmt, frame, faded(rl, alphas if len(alphas) > 1 else alphas[0]), avg=avg)
        for mode in ("out", "inplace"):
            assert_planes_equal(blend(ctx, 910, fmt, frame, mode), want, f"{alphas} {mode}")


@pytest.mark.parametrize("fmt", ["NV12", "RGB", "BGRA"])
def test_per_rectangle_values(ctx, fmt):
    check_per_rectangle_values(ctx, fmt)


@pytest.mark.parametrize("fmt", PLANAR_420)
def test_per_rectangle_values_under_chroma_averaging(averaging, fmt):
    check_per_rectangle_values(averaging, fmt, avg=True)


def check_fade_inside_one_batch(ctx, fmt, avg=False, stream=920):
    w, h, n = 1280, 720, 32
    rl = (odd_rects if avg else rects)(31, w=w)
    ctx.overlay_set_rectangles(stream, rl)
    frame = random_frame(fmt, w, h, 10)
    src = ctx.acquire(fmt, w, h)
    dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
    src.upload(frame)
    ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dsts[0].c))    # prepared at 1.0
    alphas = [(n - k) / n for k in range(n)]                      # 1.0 down to 1/32 (0 would drop the bands)
    ctx.set_batch(64, 1_000_000)
    try:
        st0 = ctx.stats()
        tickets = []
        for a, d in zip(alphas, dsts):
            ctx.overlay_set_global_alpha(stream, a)
            tickets.append(ctx.submit(stream, fmt, w, h, src.c, d.c))
        ctx.flush()
        for t in tickets:
            ctx.wait(t)
        st1 = ctx.stats()
    finally:
        ctx.set_batch(32, 200)
    assert st1["launches"] - st0["launches"] == 1
    if avg:
        # the averaged chroma of both rectangles again at each new value (BLENDSPEC section 7)
        assert st1["prepare_launches"] - st0["prepare_launches"] == 2 * (n - 1)
    else:
        assert st1["prepare_launches"] == st0["prepare_launches"]
    for k in (0, 1, 7, 16, 30, 31):
        want = expected(fmt, frame, faded(rl, alphas[k]), avg=avg, w=w, h=h)
        assert_planes_equal(dsts[k].download(), want, f"frame {k} ga={alphas[k]}")
    for f in [src] + dsts:
        f.release()


def test_fade_inside_one_batch(ctx):
    check_fade_inside_one_batch(ctx, "NV12")


@pytest.mark.parametrize("fmt", ["NV12", "I420"])
def test_fade_inside_one_batch_under_chroma_averaging(averaging, fmt):
    # a stream of its own per format: a fade prepares again for every format the stream has used
    check_fade_inside_one_batch(averaging, fmt, avg=True, stream=921 if fmt == "NV12" else 922)


def check_queued_frames(ctx, fmt, avg=False):
    rl = (odd_rects if avg else rects)(41)
    ctx.overlay_set_rectangles(930, rl)
    frame = random_frame(fmt, W, H, 11)
    src, d1, d2 = ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H)
    src.upload(frame)
    ctx.set_batch(64, 1_000_000)
    try:
        ctx.overlay_set_global_alpha(930, 0.3)
        t1 = ctx.submit(930, fmt, W, H, src.c, d1.c)
        ctx.overlay_set_global_alpha(930, 0.8)
        t2 = ctx.submit(930, fmt, W, H, src.c, d2.c)
        ctx.flush()
        ctx.wait(t1)
        ctx.wait(t2)
    finally:
        ctx.set_batch(32, 200)
    assert_planes_equal(d1.download(), expected(fmt, frame, faded(rl, 0.3), avg=avg), "first")
    assert_planes_equal(d2.download(), expected(fmt, frame, faded(rl, 0.8), avg=avg), "second")
    for f in (src, d1, d2):
        f.release()


def test_queued_frames_keep_their_alpha(ctx):
    check_queued_frames(ctx, "I420")


@pytest.mark.parametrize("fmt", ["YV12", "NV21"])
def test_queued_frames_keep_their_alpha_under_chroma_averaging(averaging, fmt):
    check_queued_frames(averaging, fmt, avg=True)


REGIONS = [wl.Region(16, 8, 160, 30, (0, 0, 0, 255), 0.8),
           wl.Region(24, 60, 150, 40, (0, 0, 128, 255), 1.0, ((255, 255, 0, 255),))]
BOXES = [(r.x, r.y, r.w, r.h) for r in REGIONS]


def region_image(seeds):
    img = np.zeros((H, W, 4), dtype=np.uint8)
    for k, (reg, seed) in enumerate(zip(REGIONS, seeds)):
        one = wl.make_overlay(W, H, [reg], 5000 + 10 * seed + k)
        img[reg.y:reg.y + reg.h, reg.x:reg.x + reg.w] = one[reg.y:reg.y + reg.h, reg.x:reg.x + reg.w]
    return img


def ttml_want(fmt, frame, img, alpha, avg=False):
    return expected(fmt, frame, faded(oracle.ttmlrender_rectangles(img), alpha), avg=avg)


def check_lifecycle(ctx, fmt, avg=False):
    frame = random_frame(fmt, W, H, 12)
    a, b = region_image([1, 1]), region_image([1, 2])
    ctx.overlay_set(940, a, BOXES)
    blend(ctx, 940, fmt, frame)
    ctx.overlay_set_global_alpha(940, [0.5, 0.5])                 # one value per region box
    assert_planes_equal(blend(ctx, 940, fmt, frame), ttml_want(fmt, frame, a, 0.5, avg), "faded")
    ctx.overlay_update(940, b, [BOXES[1]])                         # a patch keeps the value
    assert_planes_equal(blend(ctx, 940, fmt, frame), ttml_want(fmt, frame, b, 0.5, avg), "after overlay_update")
    ctx.overlay_set_global_alpha(940, [0.5, 0.25])                 # the patched box faded on its own
    assert_planes_equal(blend(ctx, 940, fmt, frame), expected(fmt, frame, regions_faded(b, [0.5, 0.25]), avg=avg),
                        "patched box faded")
    ctx.overlay_set(940, a, BOXES)                                 # a new cue starts at 1
    assert_planes_equal(blend(ctx, 940, fmt, frame), ttml_want(fmt, frame, a, 1.0, avg), "after overlay_set")

    # installed at 0.4: prepared with it folded in; the first fade prepares once more, later ones never
    rl = (odd_rects if avg else rects)(51, ga=0.4)
    st = (941 if fmt == "NV12" else 942) + (10 if avg else 0)   # a stream of its own: eager prepare adds
    ctx.overlay_set_rectangles(st, rl)                          # the formats a stream used
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, rl, avg=avg), "at 0.4")
    p0 = ctx.stats()["prepare_launches"]
    ctx.overlay_set_global_alpha(st, 0.8)
    p1 = ctx.stats()["prepare_launches"]
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, faded(rl, 0.8), avg=avg), "0.4 -> 0.8")
    ctx.overlay_set_global_alpha(st, 0.6)
    ctx.overlay_set_global_alpha(st, [0.0, 1.0])
    assert_planes_equal(blend(ctx, st, fmt, frame), expected(fmt, frame, faded(rl, [0.0, 1.0]), avg=avg), "-> 0, 1")
    p2 = ctx.stats()["prepare_launches"]
    if fmt == "BGRA":
        assert p1 == p0                 # the packed kinds never fold it in
    else:
        assert p1 > p0                  # PLANE8: the alpha bytes had 0.4 in them
    if avg:
        assert p2 > p1                  # averaged chroma holds the value: prepared again per change
    else:
        assert p2 == p1


def regions_faded(img, alphas):
    """The region image as one rectangle per region box, each at its own global alpha (the boxes
    are disjoint and the image is transparent outside them)."""
    out = []
    for (x, y, w, h), a in zip(BOXES, alphas):
        out.append(dict(pixels=np.ascontiguousarray(img[y:y + h, x:x + w]), x=x, y=y, global_alpha=a))
    return out


@pytest.mark.parametrize("fmt", ["NV12", "BGRA"])
def test_lifecycle(ctx, fmt):
    check_lifecycle(ctx, fmt)


@pytest.mark.parametrize("fmt", ["NV12", "I420"])
def test_lifecycle_under_chroma_averaging(averaging, fmt):
    check_lifecycle(averaging, fmt, avg=True)


def opaque_cue():
    """An opaque box (every pixel alpha 255) over most of the cue, and anti-aliased text."""
    box = np.zeros((64, 160, 4), dtype=np.uint8)
    box[..., :3] = (40, 80, 120)
    box[..., 3] = 255
    return [dict(pixels=box, x=16, y=16), dict(pixels=random_overlay(100, 40, 61), x=30, y=28)]


OPAQUE_CHECK = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
from test_gpu_global_alpha import check_opaque_cue
import helpers
c = helpers.pkg.TtmlBlend(0)
try:
    check_opaque_cue(c, int(sys.argv[3]))
finally:
    c.close()
print("ok")
"""


def check_opaque_cue(ctx, stream):
    for fmt in ("NV12", "RGB", "BGRA"):
        frame = random_frame(fmt, W, H, 13)
        rl = opaque_cue()
        ctx.overlay_set_rectangles(stream, rl)
        for alpha in (1.0, 0.5, 1.0, 0.0):
            ctx.overlay_set_global_alpha(stream, alpha)
            want = oracle_blend(fmt, W, H, copy_planes(frame), faded(rl, alpha))
            for mode in ("out", "inplace"):
                assert_planes_equal(blend(ctx, stream, fmt, frame, mode), want, f"{fmt} ga={alpha} {mode}")


def test_opaque_box_faded(ctx):
    ctx.overlay_set_rectangles(950, opaque_cue())
    blend(ctx, 950, "NV12", random_frame("NV12", W, H, 1), "inplace")
    st0 = ctx.stats()
    blend(ctx, 950, "NV12", random_frame("NV12", W, H, 1), "inplace")
    blend(ctx, 950, "NV12", random_frame("NV12", W, H, 1), "out")
    st1 = ctx.stats()
    on = lambda knob: os.environ.get(knob, "1") != "0" and os.environ.get("FLUC_TTMLBLEND_GROUPS", "1") != "0"
    if on("FLUC_TTMLBLEND_LAZY"):                                     # not forced off (tools/knob_matrix.sh)
        assert st1["lazy_launches"] > st0["lazy_launches"]           # the cue takes both shortcuts at 1.0
    if on("FLUC_TTMLBLEND_OPAQUE_SKIP"):
        assert st1["opaque_skip_launches"] > st0["opaque_skip_launches"]
    check_opaque_cue(ctx, 951)


@pytest.mark.parametrize("knobs", [{"FLUC_TTMLBLEND_LAZY": "1", "FLUC_TTMLBLEND_OPAQUE_SKIP": "1"},
                                   {"FLUC_TTMLBLEND_LAZY": "0", "FLUC_TTMLBLEND_OPAQUE_SKIP": "0"}])
def test_opaque_box_faded_with_forced_knobs(monkeypatch, knobs):
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    here = os.path.dirname(os.path.abspath(__file__))
    out = subprocess.run([sys.executable, "-c", OPAQUE_CHECK, here, os.path.dirname(here), "952"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout + out.stderr


def test_host_frames(ctx):
    fmt, w, h, n = "NV12", 1280, 720, 8
    # full-width rows under the cue: batches of pinned pool frames qualify for the copy engines
    rl = [dict(pixels=random_overlay(w, 40, 71), x=0, y=600), dict(pixels=random_overlay(w, 30, 72), x=0, y=80)]
    ctx.overlay_set_rectangles(960, rl)
    frames = [random_frame(fmt, w, h, 80 + i) for i in range(n)]
    pinned = [ctx.acquire(fmt, w, h, on_host=True) for _ in range(n)]

    def fill():
        for p, f in zip(pinned, frames):
            for dst, src in zip(p.host_planes(), f):
                dst[...] = src

    def check(alpha, what):
        for p, f in zip(pinned, frames):
            want = oracle_blend(fmt, w, h, copy_planes(f), faded(rl, alpha))
            assert_planes_equal([np.array(x) for x in p.host_planes()], want, what)

    try:
        for dma, alpha in ((0, 0.5), (1, 0.7)):
            ctx.set_host_dma(dma)
            ctx.overlay_set_global_alpha(960, alpha)
            fill()
            st0 = ctx.stats()
            batch = tbm.TtmlBlend.Batch([960] * n, fmt, w, h, [p.c for p in pinned], [p.c for p in pinned])
            for t in ctx.blend_host_many(batch):
                ctx.wait(t)
            ctx.sync()
            if dma:
                assert ctx.stats()["host_dma_batches"] > st0["host_dma_batches"]
            check(alpha, f"pinned, host dma {dma}")
    finally:
        ctx.set_host_dma(2)
        for p in pinned:
            p.release()
    # pageable numpy frames go through the staging threads
    ctx.overlay_set_global_alpha(960, 0.25)
    st0 = ctx.stats()
    got = copy_planes(frames[0])
    ctx.wait(ctx.blend_host(960, fmt, w, h, got))
    assert ctx.stats()["staged_frames"] > st0["staged_frames"]
    assert_planes_equal(got, oracle_blend(fmt, w, h, copy_planes(frames[0]), faded(rl, 0.25)), "pageable")
    # device frames ordered after a CUDA stream (0: the legacy default stream)
    ctx.overlay_set_global_alpha(960, 0.9)
    src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
    src.upload(frames[1])
    tk = ctx.submit_many_after(tbm.TtmlBlend.Batch([960], fmt, w, h, [src.c], [dst.c]), 0)
    ctx.wait(tk[0])
    assert_planes_equal(dst.download(), oracle_blend(fmt, w, h, copy_planes(frames[1]), faded(rl, 0.9)),
                        "submit_many_after")
    src.release()
    dst.release()


@pytest.mark.parametrize("fmt", ["NV12", "RGB", "BGRA"])
def test_zero_alpha(ctx, fmt):
    frame = random_frame(fmt, W, H, 14)
    ctx.overlay_set_rectangles(970, rects(81))
    blend(ctx, 970, fmt, frame)
    ctx.overlay_set_global_alpha(970, 0.0)
    assert_planes_equal(blend(ctx, 970, fmt, frame), frame, "out of place")
    src = ctx.acquire(fmt, W, H)
    src.upload(frame)
    ctx.sync()
    before = ctx.stats()["launches"]
    ctx.wait(ctx.submit(970, fmt, W, H, src.c, src.c))
    assert ctx.stats()["launches"] == before           # no band left: nothing to launch in place
    assert_planes_equal(src.download(), frame, "in place")
    src.release()


def test_fades_under_chroma_averaging_do_not_leak():
    """Every fade under chroma averaging prepares new chroma planes: the memory the overlay cache
    holds is back at its baseline once the cue is cleared and the work has drained."""
    import time
    c = pkg.TtmlBlend(0)
    try:
        c.set_chroma_mode(True)
        fmt = "NV12"
        frame = random_frame(fmt, W, H, 15)
        src, dst = c.acquire(fmt, W, H), c.acquire(fmt, W, H)
        src.upload(frame)
        c.sync()
        base = c.stats()["cache_bytes"]
        rl = odd_rects(101)
        c.overlay_set_rectangles(990, rl)
        for k in range(24):
            alphas = [(k % 8 + 1) / 8, ((k + 3) % 8) / 8]
            c.overlay_set_global_alpha(990, alphas)
            c.submit(990, fmt, W, H, src.c, dst.c)
        c.sync()
        assert_planes_equal(dst.download(), expected(fmt, frame, faded(rl, alphas), avg=True), "last fade")
        assert c.stats()["cache_bytes"] > base
        c.overlay_clear(990)
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


def test_errors(ctx):
    def code(stream, alphas):
        with pytest.raises(tbm.TtmlBlendError) as e:
            ctx.overlay_set_global_alpha(stream, alphas)
        return e.value.code

    assert code(980, 0.5) == tbm.ERROR_NOT_FOUND                     # no overlay yet
    ctx.overlay_set_rectangles(980, rects(91) + rects(93))            # four rectangles
    ctx.overlay_set_global_alpha(980, [0.1, 0.2, 0.3, 0.4])
    ctx.overlay_set_global_alpha(980, 0.5)
    for bad in ([0.1, 0.2], [0.1] * 5, float("nan"), -0.1, 1.5, [0.5, 0.5, float("nan"), 0.5]):
        assert code(980, bad) == tbm.ERROR_INVALID_ARGUMENT, bad
    assert ctx.lib.fluc_ttmlblend_overlay_set_global_alpha(ctx.h, 980, None, 1) == tbm.ERROR_INVALID_ARGUMENT
    assert code(980, []) == tbm.ERROR_INVALID_ARGUMENT
    ctx.overlay_clear(980)
    assert code(980, 0.5) == tbm.ERROR_NOT_FOUND
    ctx.overlay_set_regions(981, W, H, [dict(x=10, y=10, w=50, h=20, background_color=0x102030ff),
                                        dict(x=40, y=60, w=50, h=20, background_color=0x405060ff)])
    ctx.overlay_set_global_alpha(981, [0.5])                         # the regions form one image
    assert code(981, [0.5, 0.5]) == tbm.ERROR_INVALID_ARGUMENT
