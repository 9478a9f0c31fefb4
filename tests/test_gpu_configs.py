"""GPU parity at BASELINE.json's full sizes: every config's frames against the oracle
(a few frames each, the oracle takes ~0.1-0.2 s per 4K frame) plus size-independent
properties over the whole batch (in-place == out-of-place == host path, untouched bytes
outside the regions, batch == one-by-one)."""
import os

import numpy as np
import pytest

from helpers import assert_planes_equal, copy_planes, oracle_blend, pkg, random_frame, random_overlay, wl
from oracle import oracle

pytestmark = pytest.mark.gpu


def run_batch(ctx, cfg, fmt, n_frames, stream=400, inplace=False):
    srcs = [ctx.acquire(fmt, cfg.width, cfg.height) for _ in range(n_frames)]
    dsts = srcs if inplace else [ctx.acquire(fmt, cfg.width, cfg.height) for _ in range(n_frames)]
    frames = [wl.frame_for(cfg, i, fmt) for i in range(n_frames)]
    for s, f in zip(srcs, frames):
        s.upload(f)
    tickets = [ctx.submit(stream, fmt, cfg.width, cfg.height, s.c, d.c) for s, d in zip(srcs, dsts)]
    ctx.wait(tickets[-1])
    outs = [d.download() for d in dsts]
    for f in set(srcs) | set(dsts):
        f.release()
    return frames, outs


@pytest.mark.parametrize("cfg_id,fmt,n_frames,n_check", [
    (1, "I420", 4, 4), (2, "NV12", 4, 4), (3, "NV12", 32, 3),
    (4, "RGBA", 8, 2), (4, "BGRA", 8, 2), (4, "AYUV", 8, 2), (5, "I420", 8, 3),
])
def test_config_matches_oracle(ctx, cfg_id, fmt, n_frames, n_check):
    cfg = wl.CONFIGS[cfg_id]
    ov = wl.overlay_for(cfg)
    ctx.overlay_set(400, ov, wl.region_rects(cfg))
    ctx.set_batch(max(32, n_frames), 0)
    try:
        before = ctx.stats()["launches"]
        frames, outs = run_batch(ctx, cfg, fmt, n_frames)
        assert ctx.stats()["launches"] - before == 1          # the whole batch in one launch
        ref_rects = oracle.ttmlrender_rectangles(ov)
        for i in list(range(n_check - 1)) + [n_frames - 1]:
            want = oracle_blend(fmt, cfg.width, cfg.height, copy_planes(frames[i]), ref_rects)
            assert_planes_equal(outs[i], want, f"cfg {cfg_id} {fmt} frame {i}")
        # property: bytes outside the region rows are copied through untouched
        y_lo = min(r.y for r in cfg.regions)
        for fr, out in zip(frames, outs):
            assert np.array_equal(out[0][:y_lo], fr[0][:y_lo])
        # property: in place == out of place, for every frame of the batch
        _, outs_ip = run_batch(ctx, cfg, fmt, n_frames, inplace=True)
        for i, (a, b) in enumerate(zip(outs, outs_ip)):
            assert_planes_equal(b, a, f"in-place frame {i}")
    finally:
        ctx.set_batch(32, 200)


@pytest.mark.parametrize("cfg_id,fmt", [(2, "NV12"), (3, "NV12"), (4, "BGRA")])
def test_host_path_matches_device_path(ctx, cfg_id, fmt):
    """blend_host (the gst_video_overlay_composition_blend drop-in, host frames, PCIe rows
    only) gives the same bytes as the device-resident path, pinned and pageable memory."""
    cfg = wl.CONFIGS[cfg_id]
    ov = wl.overlay_for(cfg)
    ctx.overlay_set(401, ov, wl.region_rects(cfg))
    frames = [wl.frame_for(cfg, i, fmt) for i in range(3)]
    want = [oracle_blend(fmt, cfg.width, cfg.height, copy_planes(f), oracle.ttmlrender_rectangles(ov))
            for f in frames]
    # pageable numpy memory
    for f, w in zip(frames, want):
        got = copy_planes(f)
        ctx.wait(ctx.blend_host(401, fmt, cfg.width, cfg.height, got))
        assert_planes_equal(got, w, "pageable")
    # pinned pool frames, several in flight
    pinned = [ctx.acquire(fmt, cfg.width, cfg.height, on_host=True) for _ in frames]
    for p, f in zip(pinned, frames):
        for dst, src in zip(p.host_planes(), f):
            dst[...] = src
    tickets = [ctx.blend_host_frame(401, fmt, cfg.width, cfg.height, p.c) for p in pinned]
    for t in tickets:
        ctx.wait(t)
    for p, w in zip(pinned, want):
        assert_planes_equal([np.array(x) for x in p.host_planes()], w, "pinned")
        p.release()


def test_256_streams_each_with_its_own_cue(ctx):
    """Config 5's shape on one GPU: many independent streams, one frame each, one launch."""
    cfg = wl.CONFIGS[5]
    n = 24
    ctx.set_batch(64, 0)
    try:
        ovs = [wl.overlay_for(cfg, stream=s) for s in range(n)]
        for s, ov in enumerate(ovs):
            ctx.overlay_set(1000 + s, ov, wl.region_rects(cfg))
        srcs = [ctx.acquire(cfg.fmt, cfg.width, cfg.height) for _ in range(n)]
        dsts = [ctx.acquire(cfg.fmt, cfg.width, cfg.height) for _ in range(n)]
        frames = [wl.frame_for(cfg, s) for s in range(n)]
        for s_, f in zip(srcs, frames):
            s_.upload(f)
        before = ctx.stats()["launches"]
        tk = [ctx.submit(1000 + s, cfg.fmt, cfg.width, cfg.height, srcs[s].c, dsts[s].c) for s in range(n)]
        ctx.wait(tk[-1])
        assert ctx.stats()["launches"] - before == 1
        for s in (0, 7, n - 1):
            want = oracle_blend(cfg.fmt, cfg.width, cfg.height, copy_planes(frames[s]),
                                oracle.ttmlrender_rectangles(ovs[s]))
            assert_planes_equal(dsts[s].download(), want, f"stream {s}")
        for f in srcs + dsts:
            f.release()
        for s in range(n):
            ctx.overlay_clear(1000 + s)
    finally:
        ctx.set_batch(32, 200)


def test_256_streams_with_glyph_only_cues_of_different_layouts(ctx):
    """Config 5 at full size (256 x 1080p I420, one frame per stream and step) when every
    stream's cue has no background box and its own line widths: after the auto-crop the band
    lists differ per stream, and the batch travels as multi-layout launches of up to 64 frames.
    A sample of streams against the oracle, every stream against properties that need no
    oracle: rows outside the region box are copied, and blending the result's source again
    out of place gives the same bytes (the launch composition does not matter)."""
    import dataclasses
    cfg5 = wl.CONFIGS[5]
    cfg = dataclasses.replace(cfg5, regions=[dataclasses.replace(cfg5.regions[0], bg=(0, 0, 0, 0))])
    r = cfg.regions[0]
    n, distinct = 256, 48
    rng = np.random.default_rng(5)
    ovs = []
    for k in range(distinct):
        ov = wl.overlay_for(cfg, stream=k)
        ov[r.y:r.y + r.h // 2, r.x + int(rng.integers(r.w // 4, r.w)):] = 0
        ov[r.y + r.h // 2:r.y + r.h, r.x + int(rng.integers(r.w // 4, r.w)):] = 0
        ovs.append(ov)
    ctx.set_batch(256, 0)
    try:
        for s in range(n):
            ctx.overlay_set(2000 + s, ovs[s % distinct], wl.region_rects(cfg))
        base = wl.frame_for(cfg, 0)
        srcs = [ctx.acquire(cfg.fmt, cfg.width, cfg.height) for _ in range(n)]
        dsts = [ctx.acquire(cfg.fmt, cfg.width, cfg.height) for _ in range(n)]
        for s_ in srcs:
            s_.upload(base)
        ctx.sync()
        ctx.stats_reset()
        tk = ctx.submit_many(ctx.Batch([2000 + s for s in range(n)], cfg.fmt, cfg.width, cfg.height,
                                       [s_.c for s_ in srcs], [d.c for d in dsts]))
        ctx.wait(tk[n - 1])
        st = ctx.stats()
        assert st["frames_blended"] == n and st["multi_launches"] >= 4 and st["launches"] <= 8, st
        outs = {}
        for s in (0, 1, 47, 48, 100, 255):
            outs[s] = dsts[s].download()
            want = oracle_blend(cfg.fmt, cfg.width, cfg.height, copy_planes(base),
                                oracle.ttmlrender_rectangles(ovs[s % distinct]))
            assert_planes_equal(outs[s], want, f"stream {s}")
        assert_planes_equal(outs[48], outs[0], "same cue, different launch")     # 48 % 48 == 0
        for s in range(0, n, 5):
            out = outs.get(s) or dsts[s].download()
            assert np.array_equal(out[0][:r.y], base[0][:r.y]) and np.array_equal(out[0][r.y + r.h:], base[0][r.y + r.h:])
            assert np.array_equal(out[1][:r.y // 2], base[1][:r.y // 2])
            assert not np.array_equal(out[0][r.y:r.y + r.h], base[0][r.y:r.y + r.h])
            one = ctx.acquire(cfg.fmt, cfg.width, cfg.height)
            ctx.wait(ctx.submit(2000 + s, cfg.fmt, cfg.width, cfg.height, srcs[s].c, one.c))
            assert_planes_equal(one.download(), out, f"stream {s} alone vs in the batch")
            one.release()
        for f in srcs + dsts:
            f.release()
        for s in range(n):
            ctx.overlay_clear(2000 + s)
    finally:
        ctx.set_batch(32, 200)


@pytest.mark.parametrize("fmt,w,h", [("NV12", 1920, 1080), ("I420", 1279, 719), ("BGRA", 640, 360)])
def test_pinned_and_registered_host_frames_match_oracle(fmt, w, h):
    """blend_host on pinned pool frames and on host_register'ed numpy memory: the kernel reads
    and writes them over PCIe (zero copy or host DMA batches). Both equal the oracle."""
    c = pkg.TtmlBlend(0)
    try:
        rects = [dict(pixels=random_overlay(w // 2, h // 4, 5), x=w // 4 + 1, y=h // 2 + 1),
                 dict(pixels=random_overlay(w // 3, h // 5, 6), x=3, y=7, global_alpha=0.9)]
        c.overlay_set_rectangles(2, rects)
        frames = [random_frame(fmt, w, h, 40 + i) for i in range(6)]
        want = [oracle_blend(fmt, w, h, copy_planes(f), rects) for f in frames]
        pinned = [c.acquire(fmt, w, h, on_host=True) for _ in frames]
        for p, f in zip(pinned, frames):
            for dst, src in zip(p.host_planes(), f):
                dst[...] = src
        tickets = [c.blend_host_frame(2, fmt, w, h, p.c) for p in pinned]
        for t in reversed(tickets):
            c.wait(t)
        for p, wnt in zip(pinned, want):
            assert_planes_equal([np.array(x) for x in p.host_planes()], wnt, "pinned")
        st = c.stats()
        assert st["h2d_bytes"] > 0 and st["d2h_bytes"] > 0
        # registered (cudaHostRegister) numpy memory takes the same route as pool frames
        buf = np.zeros(sum(r * cw for r, cw in wl.plane_shapes(fmt, w, h)) + 4096, dtype=np.uint8)
        c.host_register(buf)
        off, planes = 0, []
        for (r, cw), src in zip(wl.plane_shapes(fmt, w, h), frames[0]):
            v = buf[off:off + r * cw].reshape(r, cw)
            v[...] = src
            planes.append(v)
            off += r * cw
        c.wait(c.blend_host(2, fmt, w, h, planes))
        assert_planes_equal(planes, want[0], "registered")
        c.sync()
        c.host_unregister(buf)
    finally:
        c.close()


def test_very_wide_frame_splits_windows(ctx):
    """A 32752-pixel-wide plane has 2047 vectors per row; the row/column division by
    multiplication is only exact up to ~2050 rows there, so the host must cut the plane into
    several windows (push_window). Checked against the oracle on the rows under the cue and
    against the source everywhere else."""
    fmt, w, h = "NV12", 32752, 2200
    rects = [dict(pixels=np.ascontiguousarray(np.tile(random_overlay(256, 24, 3), (1, 100, 1))[:, :25000]),
                  x=123, y=2100), dict(pixels=random_overlay(300, 40, 4), x=32600, y=7)]
    planes = wl.make_frame(fmt, w, h, 99)
    want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
    ctx.overlay_set_rectangles(31, rects)
    src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
    try:
        src.upload(planes)
        ctx.wait(ctx.submit(31, fmt, w, h, src.c, dst.c))
        assert_planes_equal(dst.download(), want, "wide out of place")
        ctx.wait(ctx.submit(31, fmt, w, h, src.c, src.c))
        assert_planes_equal(src.download(), want, "wide in place")
    finally:
        src.release()
        dst.release()


def test_unaligned_pinned_host_frame_is_staged(ctx):
    """Pinned host frames whose strides are not multiples of 16 must not be blended zero-copy
    (byte accesses over PCIe): their rows go through an aligned pinned staging frame (worker
    threads, then the vector kernel) and still come out right."""
    fmt, w, h = "I420", 1000, 562          # chroma stride 500: 4-byte but not 16-byte aligned
    rects = [dict(pixels=random_overlay(700, 120, 8), x=151, y=400)]
    ctx.overlay_set_rectangles(32, rects)
    planes = random_frame(fmt, w, h, 4242)
    want = oracle_blend(fmt, w, h, copy_planes(planes), rects)
    buf = np.zeros(sum(p.size for p in planes) + 64, dtype=np.uint8)
    ctx.host_register(buf)
    try:
        off, views = 0, []
        for p in planes:
            v = buf[off:off + p.size].reshape(p.shape)
            v[...] = p
            views.append(v)
            off += p.size
        ctx.sync()
        ctx.stats_reset()
        ctx.wait(ctx.blend_host(32, fmt, w, h, views))
        assert_planes_equal(views, want, "unaligned pinned")
        if os.environ.get("FLUC_TTMLBLEND_GROUPS") != "0":
            assert ctx.stats()["group_launches"] == 1   # the aligned staging frame takes the vector path
    finally:
        ctx.sync()
        ctx.host_unregister(buf)


@pytest.mark.parametrize("fmt", ("NV12", "I420", "BGRA", "AYUV"))
def test_full_size_properties_without_the_oracle(ctx, fmt):
    """Size-independent properties at 4K, no oracle involved: (1) an overlay whose alphas are
    only 0 or 255 is idempotent -- blending the result again changes nothing; (2) the same
    frame blended alone, inside a batch of 16 and in place gives identical bytes; (3) bytes
    under alpha 0 are the source bytes."""
    cfg = wl.CONFIGS[3]
    w, h = cfg.width, cfg.height
    ov = wl.overlay_for(cfg).copy()
    a = ov[:, :, 3]
    hard = np.where(a >= 128, 255, 0).astype(np.uint8)
    ov[:, :, 3] = hard
    ov[:, :, :3][hard == 0] = 0                      # valid premultiplied: colour <= alpha
    ctx.overlay_set(450, ov, wl.region_rects(cfg))
    ctx.set_batch(32, 0)
    try:
        frames = [wl.frame_for(cfg, i, fmt) for i in range(2)]
        srcs = [ctx.acquire(fmt, w, h) for _ in range(16)]
        dsts = [ctx.acquire(fmt, w, h) for _ in range(16)]
        for i, s in enumerate(srcs):
            s.upload(frames[i % 2])
        # alone
        ctx.wait(ctx.submit(450, fmt, w, h, srcs[0].c, dsts[0].c))
        alone = dsts[0].download()
        # in a batch of 16
        t = ctx.submit_many(ctx.Batch([450] * 16, fmt, w, h, [s.c for s in srcs], [d.c for d in dsts]))
        ctx.wait(max(t))
        for i in (0, 2, 14):
            assert_planes_equal(dsts[i].download(), alone, f"batch member {i}")
        # idempotence: blend the result once more, in place
        ctx.wait(ctx.submit(450, fmt, w, h, dsts[0].c, dsts[0].c))
        assert_planes_equal(dsts[0].download(), alone, "idempotent for alphas in {0, 255}")
        # alpha 0 leaves the source (luma / packed plane, pixel-exact mask)
        mask = hard == 0
        if fmt in ("NV12", "I420"):
            assert np.array_equal(alone[0][mask], frames[0][0][mask])
        else:
            px = alone[0].reshape(h, w, 4)
            assert np.array_equal(px[mask], frames[0][0].reshape(h, w, 4)[mask])
        for f in srcs + dsts:
            f.release()
    finally:
        ctx.set_batch(32, 200)


def test_auto_register_moves_pageable_frames_to_zero_copy():
    """Opt-in auto registration: pageable frames are pinned on first sight and from then on
    blended zero-copy (group launches), with identical results."""
    fmt, w, h = "NV12", 640, 360
    c = pkg.TtmlBlend(0)
    try:
        rects = [dict(pixels=random_overlay(400, 60, 3), x=100, y=250)]
        c.overlay_set_rectangles(1, rects)
        frames = [random_frame(fmt, w, h, 70 + i) for i in range(4)]
        bufs = [copy_planes(f) for f in frames]
        want = [oracle_blend(fmt, w, h, copy_planes(f), rects) for f in frames]
        for b in bufs:                                  # default: staged through pinned frames
            c.wait(c.blend_host(1, fmt, w, h, b))
        st = c.stats()
        assert st["h2d_bytes"] > 0 and st["frames_blended"] == 4
        for b, wnt in zip(bufs, want):
            assert_planes_equal(b, wnt, "staged")
        c.set_auto_register(True)
        bufs = [copy_planes(f) for f in frames]
        c.stats_reset()
        tickets = [c.blend_host(1, fmt, w, h, b) for b in bufs]
        for t in tickets:
            c.wait(t)
        assert c.stats()["group_launches"] >= 1         # zero copy now
        for b, wnt in zip(bufs, want):
            assert_planes_equal(b, wnt, "auto-registered")
        assert sum(c.host_forget(p) for b in bufs for p in b) >= 4     # they were pinned, and are not any more
        c.sync()
    finally:
        c.close()                                       # unregisters what it pinned
