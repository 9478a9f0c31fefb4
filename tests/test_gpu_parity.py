"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the
same inputs -- bit-exact (integer/byte work, tolerance 0)."""
import json
import os
import threading

import numpy as np
import pytest

from helpers import (ALL_FORMATS, PACKED, PLANAR_420, assert_planes_equal, copy_planes, gpu_blend,
                     oracle_blend, pkg, random_frame, random_overlay, wl)
from oracle import oracle

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
MODES = ("out", "inplace", "host")

CASES = [
    # w, h, [(rw, rh, x, y, global_alpha, premultiplied)], opaque dest, premultiplied dest
    (64, 48, [(32, 16, 8, 8, 1.0, True)], True, False),
    (63, 47, [(31, 15, 7, 9, 1.0, True)], True, False),
    (1279, 719, [(1000, 100, 133, 575, 1.0, True)], True, False),
    (64, 48, [(40, 30, -10, -7, 1.0, True)], True, False),
    (64, 48, [(40, 30, 40, 30, 1.0, True)], True, False),
    (33, 21, [(80, 60, -20, -20, 1.0, True)], True, False),
    (64, 48, [(1, 1, 5, 5, 1.0, True), (1, 1, 6, 6, 1.0, True), (1, 1, 63, 47, 1.0, True)], True, False),
    (200, 120, [(100, 50, 8, 8, 1.0, True), (100, 50, 60, 30, 1.0, True), (50, 90, 90, 20, 1.0, True)], True, False),
    (64, 48, [(32, 16, 8, 8, 0.5, True), (20, 20, 30, 20, 0.8, False)], True, False),
    (64, 48, [(32, 16, 8, 8, 1.0, False)], True, False),
    (64, 48, [(32, 16, 9, 7, 1.0, True)], False, False),
    (64, 48, [(32, 16, 9, 7, 0.7, True), (16, 16, 12, 10, 1.0, False)], False, True),
    (640, 360, [(640, 60, 0, 290, 1.0, True), (300, 40, 170, 10, 1.0, True)], True, False),
    (64, 48, [(30, 20, 70, 10, 1.0, True)], True, False),            # fully outside
    (64, 48, [(30, 20, 3, 3, 0.0, True)], True, False),              # global alpha 0
]


def make_rects(case):
    _, _, rects, _, _ = CASES[case]
    return [dict(pixels=random_overlay(rw, rh, 900 + 10 * case + i, premultiplied=pm),
                 x=x, y=y, global_alpha=ga, premultiplied=pm)
            for i, (rw, rh, x, y, ga, pm) in enumerate(rects)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("fmt", ALL_FORMATS)
@pytest.mark.parametrize("case", range(len(CASES)))
def test_rectangles_match_oracle(ctx, fmt, case, mode):
    w, h, _, opaque, dprem = CASES[case]
    planes = random_frame(fmt, w, h, 300 + case, opaque=opaque)
    rects = make_rects(case)
    want = oracle_blend(fmt, w, h, copy_planes(planes), rects, dprem)
    got = gpu_blend(ctx, fmt, w, h, planes, rects, mode=mode, dest_premul=dprem)
    assert_planes_equal(got, want, f"{fmt} case {case} {mode}")


@pytest.mark.parametrize("fmt", ALL_FORMATS + ("RGBx", "BGRx", "xRGB", "xBGR"))
def test_golden_fixtures(ctx, fmt):
    with open(os.path.join(GOLDEN, "manifest.json")) as f:
        manifest = json.load(f)
    hits = [v for v in manifest["vectors"] if v["format"] == fmt]
    assert hits, fmt
    for v in hits:
        z = np.load(os.path.join(GOLDEN, v["file"]))
        n = int(z["n_planes"])
        planes = [z[f"in{i}"] for i in range(n)]
        rects = [dict(pixels=z[f"rect{i}"], x=int(z["pos"][i][0]), y=int(z["pos"][i][1]),
                      global_alpha=float(z["ga"][i]), premultiplied=bool(z["premul"][i]),
                      render_width=int(z["render"][i][0]) if "render" in z else 0,
                      render_height=int(z["render"][i][1]) if "render" in z else 0)
                 for i in range(int(z["n_rects"]))]
        for mode in MODES:
            got = gpu_blend(ctx, fmt, int(z["width"]), int(z["height"]), planes, rects, mode=mode,
                            dest_premul=bool(z["dest_premul"]))
            assert_planes_equal(got, [z[f"out{i}"] for i in range(n)], f"{v['file']} {mode}")


@pytest.mark.parametrize("fmt", ("I420", "NV12", "AYUV", "BGRA"))
def test_alpha_sweep(ctx, fmt):
    """Every alpha 0..255 against every frame value 0..255 for a few overlay colours."""
    w, h = 256, 256
    planes = random_frame(fmt, w, h, 1)
    ramp = np.tile(np.arange(256, dtype=np.uint8), (256, 1))
    planes[0][:, : planes[0].shape[1]] = np.resize(ramp, planes[0].shape)
    for colour in ((255, 255, 255), (0, 0, 0), (17, 130, 241)):
        ov = np.zeros((h, w, 4), dtype=np.uint8)
        a = np.arange(256, dtype=np.uint32)[:, None] * np.ones((1, w), dtype=np.uint32)
        ov[:, :, 3] = a
        for k in range(3):
            ov[:, :, k] = (colour[k] * a + 127) // 255
        rects = [dict(pixels=ov, x=0, y=0)]
        want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
        got = gpu_blend(ctx, fmt, w, h, planes, rects, mode="out")
        assert_planes_equal(got, want, f"{fmt} sweep {colour}")


@pytest.mark.parametrize("fmt", ("NV12", "I420", "RGBA"))
def test_unaligned_strides_take_the_byte_path(ctx, fmt):
    """Strides / pointers that are not multiples of 16 (GStreamer only guarantees 4)."""
    w, h = 150, 70
    tb = pkg.ttmlblend
    rects = [dict(pixels=random_overlay(90, 40, 5), x=31, y=13)]
    planes = random_frame(fmt, w, h, 6)
    want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
    ctx.overlay_set_rectangles(3, rects)
    big = ctx.acquire(fmt, w + 64, h)      # roomy pool frame, we carve unaligned views out of it
    out = ctx.acquire(fmt, w + 64, h)
    try:
        src_f, dst_f = tb.Frame(), tb.Frame()
        host = []
        for i, (rows, rb) in enumerate(wl.plane_shapes(fmt, w, h)):
            stride = rb + 4 - (rb % 4) + 4          # multiple of 4, not of 16 in general
            host.append((rows, rb, stride))
            for f, pool in ((src_f, big), (dst_f, out)):
                f.plane[i] = pool.c.plane[i] + 4    # 4-byte aligned base
                f.stride[i] = stride
        # upload through an unaligned-view frame: build host planes with that stride
        hp = []
        for (rows, rb, stride), p in zip(host, planes):
            buf = np.zeros((rows, stride), dtype=np.uint8)
            buf[:, :rb] = p
            hp.append(buf[:, :rb])
        hsrc = tb._frame_from_arrays(hp)
        ctx._check(ctx.lib.fluc_ttmlblend_frame_upload(ctx.h, tb.FORMATS[fmt], w, h, hsrc, src_f), "up")
        ctx.wait(ctx.submit(3, fmt, w, h, src_f, dst_f))
        got = [np.zeros((rows, rb), dtype=np.uint8) for rows, rb, _ in host]
        hdst = tb._frame_from_arrays(got)
        ctx._check(ctx.lib.fluc_ttmlblend_frame_download(ctx.h, tb.FORMATS[fmt], w, h, dst_f, hdst), "down")
        assert_planes_equal(got, want, f"{fmt} unaligned out-of-place")
        ctx.wait(ctx.submit(3, fmt, w, h, src_f, src_f))
        ctx._check(ctx.lib.fluc_ttmlblend_frame_download(ctx.h, tb.FORMATS[fmt], w, h, src_f, hdst), "down")
        assert_planes_equal(got, want, f"{fmt} unaligned in place")
    finally:
        big.release()
        out.release()


@pytest.mark.parametrize("fmt", ("I420", "NV12", "BGRA", "AYUV"))
def test_ttmlrender_form_equals_whole_image(ctx, fmt):
    """overlay_set(image, region boxes) == blending the whole frame-sized image as the
    reference pipeline does, also when the region boxes overlap or leave the frame."""
    w, h = 320, 180
    regions = [wl.Region(10, 100, 300, 60, (0, 0, 0, 255), 0.7),
               wl.Region(100, 20, 150, 100, (10, 20, 200, 128), 1.0, ((255, 255, 0, 255),)),
               wl.Region(250, 150, 100, 50, (200, 0, 0, 255), 0.5)]
    ov = wl.make_overlay(w, h, regions, 77, cell=(8, 16))
    boxes = [(r.x, r.y, r.w, r.h) for r in regions]
    planes = random_frame(fmt, w, h, 8)
    want = oracle_blend(fmt, w, h, copy_planes(planes), oracle.ttmlrender_rectangles(ov))
    for mode in MODES:
        got = gpu_blend(ctx, fmt, w, h, planes, overlay=ov, regions=boxes, mode=mode)
        assert_planes_equal(got, want, f"{fmt} regions {mode}")
        got = gpu_blend(ctx, fmt, w, h, planes, overlay=ov, regions=(), mode=mode)
        assert_planes_equal(got, want, f"{fmt} whole image {mode}")


def test_clear_and_missing_overlay_pass_frames_through(ctx):
    w, h = 128, 64
    planes = random_frame("NV12", w, h, 2)
    ctx.overlay_clear(55)
    for mode in MODES:
        got = gpu_blend(ctx, "NV12", w, h, planes, mode=mode, stream=55, set_overlay=False)
        assert_planes_equal(got, planes, f"no overlay {mode}")
    ctx.overlay_set_rectangles(55, [dict(pixels=random_overlay(50, 20, 3), x=5, y=5)])
    got = gpu_blend(ctx, "NV12", w, h, planes, mode="out", stream=55, set_overlay=False)
    assert not np.array_equal(got[0], planes[0])
    ctx.overlay_clear(55)
    got = gpu_blend(ctx, "NV12", w, h, planes, mode="out", stream=55, set_overlay=False)
    assert_planes_equal(got, planes, "after clear")


def test_queued_frames_keep_the_overlay_they_were_submitted_with(ctx):
    """overlay_set replaces atomically: a frame queued before the cue change is blended with
    the old cue (the [PTS, PTS+duration) lifetime of gst_ttmlbase_gen_buffer buffers)."""
    w, h, fmt = 128, 64, "I420"
    ctx.set_batch(32, 0)
    try:
        planes = random_frame(fmt, w, h, 4)
        r_old = [dict(pixels=random_overlay(60, 30, 10), x=4, y=4)]
        r_new = [dict(pixels=random_overlay(60, 30, 11), x=40, y=20)]
        src, d0, d1 = (ctx.acquire(fmt, w, h) for _ in range(3))
        src.upload(planes)
        ctx.overlay_set_rectangles(9, r_old)
        t0 = ctx.submit(9, fmt, w, h, src.c, d0.c)
        ctx.overlay_set_rectangles(9, r_new)
        t1 = ctx.submit(9, fmt, w, h, src.c, d1.c)
        ctx.wait(t1)
        ctx.wait(t0)
        assert_planes_equal(d0.download(), oracle_blend(fmt, w, h, copy_planes(planes), r_old), "old cue")
        assert_planes_equal(d1.download(), oracle_blend(fmt, w, h, copy_planes(planes), r_new), "new cue")
        for f in (src, d0, d1):
            f.release()
    finally:
        ctx.set_batch(32, 200)


def test_mixed_batch_many_streams_one_launch(ctx):
    """Frames of different formats, sizes and streams in one batch."""
    ctx.set_batch(64, 0)
    try:
        jobs = []
        for i, (fmt, w, h) in enumerate([("NV12", 320, 180), ("I420", 200, 100), ("BGRA", 160, 90),
                                         ("AYUV", 96, 54), ("NV12", 322, 182), ("RGBA", 64, 64),
                                         ("YV12", 130, 70), ("NV21", 128, 72), ("ARGB", 50, 40)] * 3):
            planes = random_frame(fmt, w, h, 50 + i)
            rects = [dict(pixels=random_overlay(w // 2, h // 3, 60 + i), x=w // 5 + (i % 3), y=h // 2 - (i % 5))]
            ctx.overlay_set_rectangles(100 + i, rects)
            src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
            src.upload(planes)
            jobs.append((fmt, w, h, planes, rects, src, dst))
        before = ctx.stats()["launches"]
        tickets = [ctx.submit(100 + i, fmt, w, h, src.c, dst.c)
                   for i, (fmt, w, h, _, _, src, dst) in enumerate(jobs)]
        ctx.wait(tickets[-1])
        st = ctx.stats()
        assert st["launches"] - before >= 3     # at least one per plane kind
        assert st["group_launches"] > 0         # same-geometry frames share a group launch
        for fmt, w, h, planes, rects, src, dst in jobs:
            assert_planes_equal(dst.download(), oracle_blend(fmt, w, h, copy_planes(planes), rects), fmt)
            src.release()
            dst.release()
    finally:
        ctx.set_batch(32, 200)


def test_scheduler_thread_launches_partial_batches(ctx):
    """Without flush/wait the linger timer of the scheduler thread launches the batch."""
    import time
    w, h, fmt = 128, 64, "NV12"
    ctx.set_batch(32, 500)
    planes = random_frame(fmt, w, h, 12)
    rects = [dict(pixels=random_overlay(64, 32, 13), x=10, y=10)]
    ctx.overlay_set_rectangles(21, rects)
    src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
    src.upload(planes)
    before = ctx.stats()["launches"]
    ctx.submit(21, fmt, w, h, src.c, dst.c)
    deadline = time.time() + 5.0
    while ctx.stats()["launches"] == before and time.time() < deadline:
        time.sleep(0.005)
    assert ctx.stats()["launches"] == before + 1
    ctx.sync()
    assert_planes_equal(dst.download(), oracle_blend(fmt, w, h, copy_planes(planes), rects), "linger")
    src.release()
    dst.release()
    ctx.set_batch(32, 200)


def test_concurrent_submitters(ctx):
    """Many video streaming threads submit at once (one stream each)."""
    w, h, fmt, n_threads, n_frames = 160, 90, "I420", 8, 6
    results, errors = {}, []

    def worker(t):
        try:
            rects = [dict(pixels=random_overlay(100, 30, 500 + t), x=20 + t, y=40 - t)]
            ctx.overlay_set_rectangles(300 + t, rects)
            outs = []
            for i in range(n_frames):
                planes = random_frame(fmt, w, h, 1000 + 10 * t + i)
                src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
                src.upload(planes)
                tk = ctx.submit(300 + t, fmt, w, h, src.c, dst.c)
                outs.append((planes, rects, src, dst, tk))
            for planes, rects, src, dst, tk in outs:
                ctx.wait(tk)
                got = dst.download()
                want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
                assert_planes_equal(got, want, f"thread {t}")
                src.release()
                dst.release()
            results[t] = True
        except Exception as e:      # noqa: BLE001
            errors.append((t, repr(e)))

    ths = [threading.Thread(target=worker, args=(t,)) for t in range(n_threads)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    assert not errors, errors
    assert len(results) == n_threads


def test_error_codes(ctx):
    tb = pkg.ttmlblend
    f = tb.Frame()
    assert ctx.lib.fluc_ttmlblend_submit(ctx.h, 1, 99, 64, 64, 0, f, f, None) == tb.ERROR_UNSUPPORTED_FORMAT
    assert ctx.lib.fluc_ttmlblend_submit(ctx.h, 1, 0, 64, 64, 0, f, f, None) == tb.ERROR_INVALID_ARGUMENT
    assert ctx.lib.fluc_ttmlblend_wait(ctx.h, 1 << 60) == tb.ERROR_NOT_FOUND
    assert ctx.lib.fluc_ttmlblend_overlay_set(ctx.h, 1, None, 10, 10, 40, None, 0) == tb.ERROR_INVALID_ARGUMENT
    assert ctx.lib.fluc_ttmlblend_frame_pool_release(ctx.h, f) == tb.ERROR_NOT_FOUND
    # the context is still usable afterwards (errors are not sticky unless CUDA failed)
    ctx.sync()


def test_stats_count_algorithmic_bytes(ctx):
    cfg = wl.CONFIGS[1]
    ov = wl.overlay_for(cfg)
    ctx.overlay_set(70, ov, wl.region_rects(cfg))
    src, dst = ctx.acquire(cfg.fmt, cfg.width, cfg.height), ctx.acquire(cfg.fmt, cfg.width, cfg.height)
    src.upload(wl.frame_for(cfg, 0))
    ctx.sync()
    ctx.stats_reset()
    ctx.wait(ctx.submit(70, cfg.fmt, cfg.width, cfg.height, src.c, dst.c))
    st = ctx.stats()
    assert st["frames_blended"] == 1 and st["launches"] == 1
    assert st["algorithmic_bytes"] == wl.algorithmic_bytes(cfg) == 3207168
    src.release()
    dst.release()


def _text_like_overlay(w, h, seed):
    """Frame-sized image as ttmlrender emits it for transparent-background regions: a few
    lines of glyph boxes, everything else alpha 0."""
    r = np.random.default_rng(seed)
    ov = np.zeros((h, w, 4), dtype=np.uint8)
    for (y0, y1, x0, x1) in ((h // 8, h // 8 + 14, w // 4, w // 4 + w // 3),
                             (h // 8 + 20, h // 8 + 34, w // 5, w // 5 + w // 2),
                             (h - 60, h - 44, 17, w - 23), (h - 38, h - 22, w // 3, w - 101)):
        a = r.integers(1, 256, size=(y1 - y0, x1 - x0), dtype=np.uint8)
        a[r.random(a.shape) < 0.3] = 0
        c = r.integers(0, 256, size=(y1 - y0, x1 - x0, 3), dtype=np.uint8)
        ov[y0:y1, x0:x1, :3] = (c.astype(np.uint32) * a[:, :, None] // 255).astype(np.uint8)
        ov[y0:y1, x0:x1, 3] = a
    return ov


@pytest.mark.parametrize("fmt", ("I420", "NV12", "RGBA", "AYUV"))
def test_autocrop_of_sparse_frame_sized_overlay(ctx, fmt):
    """The element hands over ttmlrender's whole W x H image (no region boxes). The overlay
    cache crops it to the runs of non-transparent rows; results stay bit-exact and the
    host-frame path moves only those rows over PCIe."""
    w, h = 640, 360
    ov = _text_like_overlay(w, h, 21)
    planes = random_frame(fmt, w, h, 22)
    want = oracle_blend(fmt, w, h, copy_planes(planes), oracle.ttmlrender_rectangles(ov))
    for mode in MODES:
        got = gpu_blend(ctx, fmt, w, h, planes, overlay=ov, regions=(), mode=mode, stream=77)
        assert_planes_equal(got, want, f"{fmt} autocrop {mode}")
    pinned = ctx.acquire(fmt, w, h, on_host=True)
    for d, s in zip(pinned.host_planes(), planes):
        d[...] = s
    ctx.sync()
    ctx.stats_reset()
    ctx.wait(ctx.blend_host_frame(77, fmt, w, h, pinned.c))
    st = ctx.stats()
    frame_bytes = sum(p.size for p in planes)
    assert 0 < st["h2d_bytes"] < 0.35 * frame_bytes, (st["h2d_bytes"], frame_bytes)
    assert st["h2d_bytes"] == st["d2h_bytes"]
    assert_planes_equal([np.array(x) for x in pinned.host_planes()], want, "pinned autocrop")
    pinned.release()


def test_fully_transparent_overlay_moves_nothing(ctx):
    w, h = 320, 180
    ov = np.zeros((h, w, 4), dtype=np.uint8)
    ov[:, :, :3] = 7                      # colour without alpha: still transparent
    planes = random_frame("NV12", w, h, 23)
    for mode in MODES:
        got = gpu_blend(ctx, "NV12", w, h, planes, overlay=ov, mode=mode, stream=78)
        assert_planes_equal(got, planes, f"transparent {mode}")


def test_submit_many_equals_submit(ctx):
    """One call for a batch of frames of several streams == one submit per frame."""
    w, h, fmt, n = 256, 144, "NV12", 12
    ctx.set_batch(64, 0)
    try:
        rects = [[dict(pixels=random_overlay(128, 40, 800 + s), x=20 + 3 * s, y=60 + s)] for s in range(3)]
        for s in range(3):
            ctx.overlay_set_rectangles(600 + s, rects[s])
        frames = [random_frame(fmt, w, h, 820 + i) for i in range(n)]
        srcs = [ctx.acquire(fmt, w, h) for _ in range(n)]
        dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
        for s_, f in zip(srcs, frames):
            s_.upload(f)
        streams = [600 + (i % 3) for i in range(n)]
        batch = ctx.Batch(streams, fmt, w, h, [s_.c for s_ in srcs], [d.c for d in dsts])
        tickets = ctx.submit_many(batch)
        assert len(set(tickets)) == n and all(t > 0 for t in tickets)
        ctx.wait(max(tickets))
        for i in range(n):
            want = oracle_blend(fmt, w, h, copy_planes(frames[i]), rects[i % 3])
            assert_planes_equal(dsts[i].download(), want, f"frame {i}")
        # the same destination twice in one batch must not race: second one launches after the first
        t0 = ctx.submit(600, fmt, w, h, srcs[0].c, dsts[0].c)
        t1 = ctx.submit(601, fmt, w, h, dsts[0].c, dsts[0].c)     # in place on the first result
        ctx.wait(t1)
        step1 = oracle_blend(fmt, w, h, copy_planes(frames[0]), rects[0])
        want = oracle_blend(fmt, w, h, step1, rects[1])
        assert_planes_equal(dsts[0].download(), want, "same buffer twice")
        for f in srcs + dsts:
            f.release()
    finally:
        ctx.set_batch(32, 200)


@pytest.mark.parametrize("fmt", ("NV12", "I420", "BGRA"))
@pytest.mark.parametrize("xoff,w", [(64, 320), (4, 310), (32, 333)])
def test_no_byte_outside_the_frame_is_written(ctx, fmt, xoff, w):
    """Guard-band check (compute-sanitizer is not available on the pool): the destination is a
    window inside a larger buffer; everything around it must keep its pattern, for aligned
    windows (vector path), 4-byte aligned ones (byte path) and ragged widths."""
    tb = pkg.ttmlblend
    h, W2, H2, yoff = 90, 512, 128, 10
    rects = [dict(pixels=random_overlay(w + 40, 50, 31), x=-20, y=30),
             dict(pixels=random_overlay(60, 200, 32), x=w - 30, y=-50)]
    ctx.overlay_set_rectangles(88, rects)
    planes = random_frame(fmt, w, h, 33)
    want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
    big_src, big_dst = ctx.acquire(fmt, W2, H2), ctx.acquire(fmt, W2, H2)
    try:
        pattern = [np.full((rows, rb), 0xA5, dtype=np.uint8) for rows, rb in wl.plane_shapes(fmt, W2, H2)]
        big_dst.upload(pattern)
        big_src.upload(pattern)
        bpp = 4 if fmt == "BGRA" else 1
        src_f, dst_f, views = tb.Frame(), tb.Frame(), []
        for i, ((rows, rb), (_, rb_big)) in enumerate(zip(wl.plane_shapes(fmt, w, h), wl.plane_shapes(fmt, W2, H2))):
            sub = 1 if i == 0 or fmt == "BGRA" else 2                 # chroma subsampling of the offsets
            xo = (xoff // sub) * bpp if not (fmt == "NV12" and i == 1) else xoff     # NV12 UV: 2 bytes per 2 px
            yo = yoff // sub
            for f, pool in ((src_f, big_src), (dst_f, big_dst)):
                f.plane[i] = pool.c.plane[i] + yo * pool.c.stride[i] + xo
                f.stride[i] = pool.c.stride[i]
            views.append((yo, xo, rows, rb))
        host = tb._frame_from_arrays([np.ascontiguousarray(p) for p in planes])
        ctx._check(ctx.lib.fluc_ttmlblend_frame_upload(ctx.h, tb.FORMATS[fmt], w, h, host, src_f), "up")
        for s_frame, d_frame, what in ((src_f, dst_f, "out of place"), (dst_f, dst_f, "in place again")):
            if what == "in place again":       # restore the unblended frame inside the window first
                ctx._check(ctx.lib.fluc_ttmlblend_frame_upload(ctx.h, tb.FORMATS[fmt], w, h, host, dst_f), "up")
            ctx.wait(ctx.submit(88, fmt, w, h, s_frame, d_frame))
            got_big = big_dst.download()
            for (yo, xo, rows, rb), g, wnt in zip(views, got_big, want):
                assert np.array_equal(g[yo:yo + rows, xo:xo + rb], wnt), what
                outside = g.copy()
                outside[yo:yo + rows, xo:xo + rb] = 0xA5
                assert (outside == 0xA5).all(), f"{what}: {int((outside != 0xA5).sum())} guard bytes overwritten"
    finally:
        big_src.release()
        big_dst.release()


def test_stress_cue_changes_while_frames_flow(ctx):
    """Subtitle threads replace cues while video threads submit device frames and host frames
    of the same streams: every frame must equal the oracle for the cue that was current at
    submit time (atomic replace), whatever batches the scheduler forms."""
    w, h, fmt, n_streams, rounds = 192, 108, "NV12", 6, 12
    ctx.set_batch(16, 100)
    errors = []
    cues = [[dict(pixels=random_overlay(120, 30, 7000 + 10 * s + k), x=10 + 5 * k, y=20 + 7 * k + s)]
            for s in range(n_streams) for k in range(2)]

    def stream_thread(s):
        try:
            src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
            pinned = ctx.acquire(fmt, w, h, on_host=True)
            for r in range(rounds):
                cue = cues[2 * s + (r & 1)]
                ctx.overlay_set_rectangles(900 + s, cue)
                planes = random_frame(fmt, w, h, 7100 + 100 * s + r)
                want = oracle_blend(fmt, w, h, copy_planes(planes), cue)
                src.upload(planes)
                t_dev = ctx.submit(900 + s, fmt, w, h, src.c, dst.c)
                for d, p in zip(pinned.host_planes(), planes):
                    d[...] = p
                t_host = ctx.blend_host_frame(900 + s, fmt, w, h, pinned.c)
                if r % 3 == 0:
                    ctx.overlay_clear(900 + s)          # must not affect the two frames above
                ctx.wait(t_host)
                ctx.wait(t_dev)
                assert_planes_equal(dst.download(), want, f"stream {s} round {r} device")
                assert_planes_equal([np.array(x) for x in pinned.host_planes()], want,
                                    f"stream {s} round {r} host")
            for f in (src, dst, pinned):
                f.release()
        except Exception as e:      # noqa: BLE001
            errors.append((s, repr(e)))

    ths = [threading.Thread(target=stream_thread, args=(s,)) for s in range(n_streams)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    ctx.set_batch(32, 200)
    assert not errors, errors


@pytest.mark.parametrize("seed", range(40))
def test_fuzz_random_geometry(ctx, seed):
    """Seeded fuzz over everything the host-side job builder has to cut correctly: odd and
    tiny frames, many rectangles hanging over every border or overlapping, sparse and dense
    overlays, global alpha, straight / premultiplied sources, non-opaque and premultiplied
    destinations, all formats and all three ways into the library."""
    r = np.random.default_rng(9000 + seed)
    fmt = ALL_FORMATS[seed % len(ALL_FORMATS)]
    w = int(r.choice([r.integers(1, 40), r.integers(40, 400), 16 * r.integers(1, 30)]))
    h = int(r.choice([r.integers(1, 30), r.integers(30, 200)]))
    packed = fmt in PACKED
    opaque = bool(r.random() < 0.7) or not packed
    dprem = packed and bool(r.random() < 0.2)
    rects = []
    for i in range(int(r.integers(1, 7))):
        rw, rh = int(r.integers(1, max(2, w + 20))), int(r.integers(1, max(2, h + 20)))
        ov = random_overlay(rw, rh, int(r.integers(1 << 30)), premultiplied=bool(r.random() < 0.7),
                            density=float(r.choice([0.05, 0.5, 1.0])))
        if r.random() < 0.3:
            ov[:, :, 3][r.random((rh, rw)) < 0.9] = 0          # mostly transparent: exercises the crop
            ov[:, :, :3] = np.minimum(ov[:, :, :3], ov[:, :, 3:4])
        rects.append(dict(pixels=ov, x=int(r.integers(-rw, w + 5)), y=int(r.integers(-rh, h + 5)),
                          global_alpha=float(r.choice([1.0, 1.0, 0.5, 0.99, 0.0])),
                          premultiplied=bool(r.random() < 0.7)))
    planes = random_frame(fmt, w, h, int(r.integers(1 << 30)), opaque=opaque)
    want = oracle_blend(fmt, w, h, copy_planes(planes), rects, dprem)
    for mode in MODES:
        got = gpu_blend(ctx, fmt, w, h, planes, rects, mode=mode, dest_premul=dprem, stream=40 + seed)
        assert_planes_equal(got, want, f"seed {seed} {fmt} {w}x{h} {mode}")


@pytest.mark.parametrize("fmt,w,h,with_cue", [("BGRA", 32, 32, False), ("BGRA", 64, 64, True),
                                               ("NV12", 64, 32, True), ("I420", 16, 16, False)])
def test_many_tiny_frames_in_one_group(ctx, fmt, w, h, with_cue):
    """Frames of one or a few chunks each, many per group launch (one chunk per frame is a
    corner of the frame-index arithmetic)."""
    n = 48
    ctx.set_batch(64, 0)
    try:
        rects = [dict(pixels=random_overlay(w, h // 2, 77), x=0, y=h // 4)] if with_cue else []
        if with_cue:
            ctx.overlay_set_rectangles(66, rects)
        else:
            ctx.overlay_clear(66)
        frames = [random_frame(fmt, w, h, 6000 + i) for i in range(n)]
        srcs = [ctx.acquire(fmt, w, h) for _ in range(n)]
        dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
        for s_, f in zip(srcs, frames):
            s_.upload(f)
        before = ctx.stats()
        tickets = ctx.submit_many(ctx.Batch([66] * n, fmt, w, h, [s_.c for s_ in srcs], [d.c for d in dsts]))
        ctx.wait(max(tickets))
        after = ctx.stats()
        assert after["group_launches"] - before["group_launches"] == 1
        for i in range(n):
            want = oracle_blend(fmt, w, h, copy_planes(frames[i]), rects)
            assert_planes_equal(dsts[i].download(), want, f"tiny frame {i}")
        for f in srcs + dsts:
            f.release()
    finally:
        ctx.set_batch(32, 200)


@pytest.mark.parametrize("fmt", PLANAR_420)
@pytest.mark.parametrize("w,h,rect", [(64, 48, (31, 15, 7, 9)), (63, 47, (40, 30, -10, -7)),
                                      (200, 120, (150, 60, 33, 41)), (33, 21, (80, 60, -20, -20))])
def test_chroma_average_option_is_what_it_says(fmt, w, h, rect):
    """fluc_ttmlblend_set_chroma_mode (AVERAGE): an explicit NON-PARITY option (GStreamer sites
    chroma on the even pixel). Checked against its own numpy model; luma stays bit-exact with
    the oracle, and the default mode is untouched."""
    from helpers import model_blend
    rw, rh, x, y = rect
    rects = [dict(pixels=random_overlay(rw, rh, 51), x=x, y=y),
             dict(pixels=random_overlay(20, 10, 52, premultiplied=False), x=w // 2, y=h // 3,
                  premultiplied=False, global_alpha=0.8)]
    planes = random_frame(fmt, w, h, 53)
    c = pkg.TtmlBlend(0)
    try:
        c.set_chroma_mode(True)
        want = model_blend(fmt, w, h, copy_planes(planes), rects, chroma_average=True)
        sited = oracle_blend(fmt, w, h, copy_planes(planes), rects)
        for mode in MODES:
            got = gpu_blend(c, fmt, w, h, planes, rects, mode=mode)
            assert_planes_equal(got, want, f"{fmt} average {mode}")
            assert np.array_equal(got[0], sited[0])                 # luma is not affected
        c.set_chroma_mode(False)
        c.overlay_set_rectangles(1, rects)
        got = gpu_blend(c, fmt, w, h, planes, rects, mode="out")
        assert_planes_equal(got, sited, f"{fmt} back to sited")
        assert c.lib.fluc_ttmlblend_set_chroma_mode(c.h, 7) == pkg.ttmlblend.ERROR_INVALID_ARGUMENT
    finally:
        c.close()


def test_overlay_cache_does_not_leak():
    """Hundreds of cue changes in every form (images, rectangles, regions, several formats and
    sizes, clears) with frames in between: the device memory held by the overlay caches goes
    back to zero once the cues are cleared and the work has drained."""
    c = pkg.TtmlBlend(0)
    try:
        c.sync()
        base = c.stats()["cache_bytes"]
        w, h = 320, 180
        frames = {fmt: (c.acquire(fmt, w, h), c.acquire(fmt, w, h)) for fmt in ("NV12", "I420", "BGRA", "AYUV")}
        peak = 0
        for i in range(150):
            s_id = i % 5
            if i % 3 == 0:
                c.overlay_set(s_id, random_overlay(w, h, 100 + i), [(10, 20 + i % 30, 200, 60)])
            elif i % 3 == 1:
                c.overlay_set_rectangles(s_id, [dict(pixels=random_overlay(100, 40, 200 + i), x=i % 50, y=i % 90),
                                                dict(pixels=random_overlay(60, 60, 300 + i), x=150, y=40)])
            else:
                c.overlay_set_regions(s_id, w, h, [dict(x=5, y=5 + i % 20, w=200, h=50,
                                                       background_color=0x102030C0, opacity=0.5,
                                                       layer=random_overlay(200, 50, 400 + i))])
            for fmt, (src, dst) in frames.items():
                if (i + len(fmt)) % 2:
                    c.submit(s_id, fmt, w, h, src.c, dst.c)
            if i % 7 == 0:
                c.overlay_clear((i + 2) % 5)
            if i % 10 == 0:
                peak = max(peak, c.stats()["cache_bytes"])
        c.sync()
        assert peak > base
        for s_id in range(5):
            c.overlay_clear(s_id)
        c.sync()
        c.sync()        # deferred frees run on the reaper stream after the fences
        import time
        deadline = time.time() + 5
        while c.stats()["cache_bytes"] > base and time.time() < deadline:
            time.sleep(0.01)
        assert c.stats()["cache_bytes"] == base, (c.stats()["cache_bytes"], base, peak)
    finally:
        c.close()


@pytest.mark.parametrize("fmt,twin", [("RGBx", "RGBA"), ("BGRx", "BGRA"), ("xRGB", "ARGB"), ("xBGR", "ABGR")])
def test_padded_rgb_formats_are_their_alpha_twins(ctx, fmt, twin):
    """RGBx / BGRx / xRGB / xBGR share pack/unpack with RGBA / BGRA / ARGB / ABGR in GStreamer's
    format table, so gst_video_blend treats the padding byte as destination alpha: same bytes
    out, also when the padding is not 255."""
    w, h = 200, 90
    rects = [dict(pixels=random_overlay(120, 50, 17), x=33, y=21)]
    for opaque in (True, False):
        planes = random_frame(twin, w, h, 18, opaque=opaque)
        want = oracle_blend(twin, w, h, copy_planes(planes), rects)
        assert_planes_equal(oracle_blend(fmt, w, h, copy_planes(planes), rects), want, "oracle alias")
        for mode in MODES:
            got = gpu_blend(ctx, fmt, w, h, planes, rects, mode=mode, stream=44)
            assert_planes_equal(got, want, f"{fmt} {mode} opaque={opaque}")


@pytest.mark.parametrize("fmt", ("NV12", "I420", "BGRA", "AYUV", "YUY2"))
def test_sparse_cues_take_the_overlay_first_path_in_place(ctx, fmt):
    """In place (device frames with dst == src, pinned host frames) under a cue without a
    background box the group kernel reads the overlay first and neither loads nor stores the
    vectors whose alpha is zero everywhere. Same bytes as the oracle; a cue with a filled box
    keeps the eager variant."""
    cfg = wl.CONFIGS[1]                            # 720p, one cue, transparent background
    w, h = cfg.width, cfg.height
    sparse = wl.overlay_for(cfg)
    boxed = sparse.copy()
    r = cfg.regions[0]
    box = boxed[r.y:r.y + r.h, r.x:r.x + r.w]
    box[box[..., 3] == 0] = (0, 0, 0, 96)          # a translucent black box behind the glyphs
    # an opaque box: the result under it does not depend on the frame, which is then not even
    # read (the poisoned-source check below cannot tell, the oracle comparison can: any stale
    # or garbage source byte leaking into the output would differ)
    opaque = sparse.copy()
    box = opaque[r.y:r.y + r.h, r.x:r.x + r.w]
    box[box[..., 3] == 0] = (16, 16, 16, 255)
    planes = random_frame(fmt, w, h, 3)
    for name, ov, lazy in (("sparse", sparse, True), ("boxed", boxed, False), ("opaque box", opaque, True)):
        want = oracle_blend(fmt, w, h, copy_planes(planes), oracle.ttmlrender_rectangles(ov))
        ctx.overlay_set(5, ov, wl.region_rects(cfg))
        for on_host in (False, True):
            fr = ctx.acquire(fmt, w, h, on_host=on_host)
            if on_host:
                for d, s in zip(fr.host_planes(), planes):
                    d[...] = s
            else:
                fr.upload(planes)
            ctx.sync()
            ctx.stats_reset()
            if on_host:
                ctx.wait(ctx.blend_host_frame(5, fmt, w, h, fr.c))
                got = [np.array(p) for p in fr.host_planes()]
            else:
                ctx.wait(ctx.submit(5, fmt, w, h, fr.c, fr.c))
                got = fr.download()
            st = ctx.stats()
            # which variant ran is a property of the default configuration; under a knob that
            # forces another code path (tools/knob_matrix.sh) only the bytes are checked
            if not any(k in os.environ for k in ("FLUC_TTMLBLEND_LAZY", "FLUC_TTMLBLEND_GROUPS", "FLUC_TTMLBLEND_AUTOCROP")):
                assert (st["lazy_launches"] > 0) == lazy, (name, on_host, st)
                assert st["lazy_launches"] <= st["group_launches"]
            assert_planes_equal(got, want, f"{fmt} {name} host={on_host}")
            fr.release()
        # out of place never skips a store: every byte of dst must be written. Under an opaque box
        # the frame is not read (the overlay is looked at first there too)
        got = gpu_blend(ctx, fmt, w, h, planes, mode="out", stream=5, set_overlay=False)
        st_out = ctx.stats()
        assert st_out["lazy_launches"] == (st["lazy_launches"])
        if not any(k in os.environ for k in ("FLUC_TTMLBLEND_OPAQUE_SKIP", "FLUC_TTMLBLEND_GROUPS", "FLUC_TTMLBLEND_AUTOCROP")):
            assert (st_out["opaque_skip_launches"] > st["opaque_skip_launches"]) == (name == "opaque box"), (name, st_out)
        assert_planes_equal(got, want, f"{fmt} {name} out of place")


@pytest.mark.parametrize("fmt,mode", [("I420", "out"), ("NV12", "inplace"), ("BGRA", "out"), ("AYUV", "host")])
def test_streams_with_different_cue_layouts_share_one_launch(ctx, fmt, mode):
    """Many streams of one frame geometry, each showing its own cue (other rows, other widths):
    their band lists differ, so they cannot share a plain group launch; they travel as one
    multi-layout launch (distinct band lists + per-frame layout index in the kernel parameters).
    Streams 2k and 2k+1 show the same cue and must share a band list."""
    w, h, n = 256, 144, 40
    ctx.set_batch(64, 0)
    try:
        frames, rects_of = [], []
        for i in range(n):
            k = i // 2
            rects = [dict(pixels=random_overlay(64 + 16 * (k % 9), 10 + k, 3000 + k), x=16 * (k % 5), y=8 + 3 * k)]
            if k % 3 == 0:
                rects.append(dict(pixels=random_overlay(48, 12, 3100 + k, premultiplied=False), x=100 + k, y=4,
                                  premultiplied=False, global_alpha=0.5))
            ctx.overlay_set_rectangles(500 + i, rects)
            rects_of.append(rects)
            frames.append(random_frame(fmt, w, h, 4000 + i))
        on_host = mode == "host"
        srcs = [ctx.acquire(fmt, w, h, on_host=on_host) for _ in range(n)]
        dsts = srcs if mode != "out" else [ctx.acquire(fmt, w, h) for _ in range(n)]
        for s_, f in zip(srcs, frames):
            if on_host:
                for d, p in zip(s_.host_planes(), f):
                    d[...] = p
            else:
                s_.upload(f)
        ctx.sync()
        ctx.stats_reset()
        if on_host:
            tickets = [ctx.blend_host_frame(500 + i, fmt, w, h, srcs[i].c) for i in range(n)]
        else:
            tickets = ctx.submit_many(ctx.Batch([500 + i for i in range(n)], fmt, w, h,
                                                [s_.c for s_ in srcs], [d.c for d in dsts]))
        ctx.wait(max(tickets))
        st = ctx.stats()
        assert st["multi_launches"] == 1 and st["launches"] == 1, st
        for i in range(n):
            want = oracle_blend(fmt, w, h, copy_planes(frames[i]), rects_of[i])
            got = [np.array(p) for p in dsts[i].host_planes()] if on_host else dsts[i].download()
            assert_planes_equal(got, want, f"{fmt} {mode} stream {i}")
        for f in set(srcs + dsts):
            f.release()
        for i in range(n):
            ctx.overlay_clear(500 + i)
    finally:
        ctx.set_batch(32, 200)


def test_blend_host_many_equals_blend_host(ctx):
    """One C call for a run of host frames: pinned pool frames (zero copy) and, through the
    same call, pageable numpy frames (staging threads) -- each must equal the oracle."""
    fmt, w, h, n = "NV12", 320, 180, 6
    rects = [dict(pixels=random_overlay(200, 40, 61), x=60, y=120)]
    ctx.overlay_set_rectangles(9, rects)
    frames = [random_frame(fmt, w, h, 700 + i) for i in range(n)]
    pinned = [ctx.acquire(fmt, w, h, on_host=True) for _ in range(n)]
    for hf, f in zip(pinned, frames):
        for d, p in zip(hf.host_planes(), f):
            d[...] = p
    tickets = ctx.blend_host_many(ctx.Batch([9] * n, fmt, w, h, [hf.c for hf in pinned], [hf.c for hf in pinned]))
    ctx.wait(tickets[n - 1])
    for i in range(n):
        want = oracle_blend(fmt, w, h, copy_planes(frames[i]), rects)
        assert_planes_equal([np.array(p) for p in pinned[i].host_planes()], want, f"pinned {i}")
    pageable = [copy_planes(f) for f in frames]
    cfr = [pkg.ttmlblend._frame_from_arrays(p) for p in pageable]
    tickets = ctx.blend_host_many(ctx.Batch([9] * n, fmt, w, h, cfr, cfr))
    for t in tickets:
        ctx.wait(t)
    for i in range(n):
        want = oracle_blend(fmt, w, h, copy_planes(frames[i]), rects)
        assert_planes_equal(pageable[i], want, f"pageable {i}")
    for hf in pinned:
        hf.release()


def test_layout_cache_eviction_with_frames_queued(ctx):
    """A prepared overlay keeps at most 8 layouts (one per stride / alignment combination) and
    the context at most 16 format/size entries for frames without an overlay; building one more
    while frames that use the oldest are still queued must launch those first. Twelve stride
    combinations in ONE batch, with and without an overlay, plus twenty frame sizes."""
    tb = pkg.ttmlblend
    fmt, w, h = "GRAY8", 256, 32
    rects = [dict(pixels=random_overlay(120, 16, 9), x=40, y=8)]
    big_src = ctx.acquire(fmt, 8192, 64)
    big_dst = ctx.acquire(fmt, 8192, 64)
    ctx.set_batch(64, 0)
    try:
        for stream, with_cue in ((41, True), (42, False)):
            if with_cue:
                ctx.overlay_set_rectangles(stream, rects)
            else:
                ctx.overlay_clear(stream)
            planes = random_frame(fmt, w, h, 31)
            want = oracle_blend(fmt, w, h, copy_planes(planes), rects if with_cue else [])
            strides = [256 + 16 * k for k in range(12)]            # 12 layouts, 4 of them misaligned below
            views = []
            for k, stride in enumerate(strides):
                off = 16 * k + (4 if k % 3 == 2 else 0)            # every third frame 4-byte aligned only
                sf, df = tb.Frame(), tb.Frame()
                sf.plane[0] = big_src.c.plane[0] + off
                df.plane[0] = big_dst.c.plane[0] + off
                sf.stride[0] = df.stride[0] = stride
                views.append((sf, df))
            hsrc = tb._frame_from_arrays(planes)
            # the views overlap in memory, so one at a time: upload, queue, and only then wait
            for sf, df in views:
                ctx._check(ctx.lib.fluc_ttmlblend_frame_upload(ctx.h, tb.FORMATS[fmt], w, h, hsrc, sf), "up")
                t = ctx.submit(stream, fmt, w, h, sf, df)
                ctx.wait(t)
                got = [np.zeros((h, w), dtype=np.uint8)]
                ctx._check(ctx.lib.fluc_ttmlblend_frame_download(ctx.h, tb.FORMATS[fmt], w, h, df,
                                                                 tb._frame_from_arrays(got)), "down")
                assert_planes_equal(got, want, f"stride {sf.stride[0]} cue={with_cue}")
            # and all twelve queued together, each view in its own piece of the big buffer
            views, base = [], 0
            for k, stride in enumerate(strides):
                sf, df = tb.Frame(), tb.Frame()
                off = base + (4 if k % 3 == 2 else 0)
                sf.plane[0] = big_src.c.plane[0] + off
                df.plane[0] = big_dst.c.plane[0] + off
                sf.stride[0] = df.stride[0] = stride
                views.append((sf, df))
                base += (stride * h + 4 + 255) // 256 * 256
            assert base <= 8192 * 64
            for sf, df in views:
                ctx._check(ctx.lib.fluc_ttmlblend_frame_upload(ctx.h, tb.FORMATS[fmt], w, h, hsrc, sf), "up")
            tickets = [ctx.submit(stream, fmt, w, h, sf, df) for sf, df in views]
            ctx.wait(max(tickets))
            for sf, df in views:
                got = [np.zeros((h, w), dtype=np.uint8)]
                ctx._check(ctx.lib.fluc_ttmlblend_frame_download(ctx.h, tb.FORMATS[fmt], w, h, df,
                                                                 tb._frame_from_arrays(got)), "down")
                assert_planes_equal(got, want, f"queued together, stride {sf.stride[0]} cue={with_cue}")
        # twenty sizes without an overlay, all queued before the first wait
        ctx.overlay_clear(43)
        jobs = []
        for k in range(20):
            ww, hh = 64 + 16 * k, 16 + k
            p = random_frame(fmt, ww, hh, 900 + k)
            s_, d_ = ctx.acquire(fmt, ww, hh), ctx.acquire(fmt, ww, hh)
            s_.upload(p)
            jobs.append((ctx.submit(43, fmt, ww, hh, s_.c, d_.c), p, s_, d_))
        for t, p, s_, d_ in jobs:
            ctx.wait(t)
            assert_planes_equal(d_.download(), p, "pass-through")
            s_.release()
            d_.release()
    finally:
        ctx.set_batch(32, 200)
        big_src.release()
        big_dst.release()


def test_synchronous_callers_of_many_streams_share_launches(ctx):
    """What a GStreamer process with many ttmlblend elements does: every element's streaming
    thread calls blend (host frame, in place) and waits for it, frame after frame. With several
    streams active a wait lets the batch linger (up to the linger time) instead of launching
    its own frame alone, so frames of different threads share launches; a single stream is
    launched at once. Bit-exact either way."""
    w, h, fmt, n_threads, n_frames = 320, 180, "NV12", 12, 25
    errors = []
    ctx.set_batch(32, 2000)                    # 2 ms linger: generous for Python threads
    barrier = threading.Barrier(n_threads)

    def worker(t):
        try:
            rects = [dict(pixels=random_overlay(200, 40, 800 + t), x=40 + t, y=100 + t)]
            ctx.overlay_set_rectangles(700 + t, rects)
            planes = random_frame(fmt, w, h, 2000 + t)
            want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
            hf = ctx.acquire(fmt, w, h, on_host=True)
            barrier.wait()
            for i in range(n_frames):
                for d, p in zip(hf.host_planes(), planes):
                    d[...] = p
                ctx.wait(ctx.blend_host_frame(700 + t, fmt, w, h, hf.c))
                assert_planes_equal([np.array(p) for p in hf.host_planes()], want, f"thread {t} frame {i}")
            hf.release()
        except Exception as e:      # noqa: BLE001
            errors.append((t, repr(e)))

    try:
        ctx.sync()
        ctx.stats_reset()
        ths = [threading.Thread(target=worker, args=(t,)) for t in range(n_threads)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        assert not errors, errors
        st = ctx.stats()
        assert st["frames_blended"] == n_threads * n_frames
        assert st["launches"] < 0.85 * st["frames_blended"], st         # frames did share launches
        # one stream alone is not made to wait: a launch per frame, no lingering
        ctx.stats_reset()
        import time
        rects = [dict(pixels=random_overlay(200, 40, 899), x=40, y=100)]
        ctx.overlay_set_rectangles(799, rects)
        hf = ctx.acquire(fmt, w, h, on_host=True)
        for _ in range(20):                       # the other streams drop out of the recent list
            ctx.wait(ctx.blend_host_frame(799, fmt, w, h, hf.c))
        t0 = time.perf_counter()
        for _ in range(50):
            ctx.wait(ctx.blend_host_frame(799, fmt, w, h, hf.c))
        per_frame = (time.perf_counter() - t0) / 50
        assert per_frame < 1e-3, per_frame          # far below the 2 ms linger
        hf.release()
    finally:
        ctx.set_batch(32, 200)


def test_next_cue_is_prepared_at_the_cue_change(ctx):
    """overlay_set prepares the new cue for the format / size the stream's frames have been
    using, so the first frame after a cue change launches no prepare kernel; a format the
    stream never used is not prepared ahead."""
    fmt, w, h = "NV12", 320, 180
    planes = random_frame(fmt, w, h, 8)
    src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
    src.upload(planes)
    ctx.overlay_clear(9731)                            # a stream no other test has touched
    for k in range(3):
        rects = [dict(pixels=random_overlay(200, 40, 70 + k), x=60, y=100 + k)]
        ctx.sync()
        ctx.stats_reset()
        ctx.overlay_set_rectangles(9731, rects)
        at_cue = ctx.stats()["prepare_launches"]
        ctx.wait(ctx.submit(9731, fmt, w, h, src.c, dst.c))
        at_frame = ctx.stats()["prepare_launches"] - at_cue
        if k == 0:
            assert at_cue == 0 and at_frame > 0          # nothing known about the stream yet
        else:
            assert at_cue > 0 and at_frame == 0, (k, at_cue, at_frame)
        want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
        assert_planes_equal(dst.download(), want, f"cue {k}")
    src.release()
    dst.release()


def test_cue_pixels_already_in_device_memory(ctx):
    """overlay_set / overlay_set_rectangles accept pixels that are in HBM already (a cue left
    there by a previous GPU stage): same result, and nothing counted as host -> device."""
    tb = pkg.ttmlblend
    w, h = 320, 180
    px = random_overlay(200, 40, 77)
    holder = ctx.acquire("BGRA", 200, 40)              # a device BGRA surface to put the cue in
    holder.upload([px.reshape(40, 800)])
    ctx.sync()
    ctx.stats_reset()
    arr = (tb.Rectangle * 1)(tb.Rectangle(holder.c.plane[0], 200, 40, holder.c.stride[0], 60, 100, 1.0,
                                          tb.FLAG_PREMULTIPLIED_ALPHA, 0, 0))
    ctx._check(ctx.lib.fluc_ttmlblend_overlay_set_rectangles(ctx.h, 9801, arr, 1), "overlay_set_rectangles")
    assert ctx.stats()["h2d_bytes"] == 0
    for fmt in ("NV12", "BGRA"):
        planes = random_frame(fmt, w, h, 9)
        want = oracle_blend(fmt, w, h, copy_planes(planes), [dict(pixels=px, x=60, y=100)])
        got = gpu_blend(ctx, fmt, w, h, planes, mode="out", stream=9801, set_overlay=False)
        assert_planes_equal(got, want, f"device cue {fmt}")
    # scaled, too
    arr[0].render_width, arr[0].render_height = 260, 33
    ctx._check(ctx.lib.fluc_ttmlblend_overlay_set_rectangles(ctx.h, 9801, arr, 1), "overlay_set_rectangles")
    planes = random_frame("I420", w, h, 10)
    want = oracle_blend("I420", w, h, copy_planes(planes), [dict(pixels=px, x=60, y=100, render_width=260,
                                                                  render_height=33)])
    got = gpu_blend(ctx, "I420", w, h, planes, mode="out", stream=9801, set_overlay=False)
    assert_planes_equal(got, want, "device cue, scaled")
    holder.release()
    ctx.overlay_clear(9801)
