"""Frames of one batch that depend on each other: chained overlays (stream A's output is
stream B's input), ping-pong buffers, the same buffer written twice, two overlays on one host
frame. The CTAs of one launch run in no order, so the runtime must cut the batch at such
frames; the result must equal the sequential composition computed by the oracle."""
import os

import numpy as np
import pytest

from helpers import assert_planes_equal, copy_planes, oracle_blend, pkg, random_frame, random_overlay, wl
from oracle import oracle

pytestmark = pytest.mark.gpu

W, H = 640, 360


def _overlays(n, seed):
    return [random_overlay(W, H, seed + i, density=0.5) for i in range(n)]


def _rects(ov):
    return [dict(pixels=ov, x=0, y=0)]


@pytest.mark.parametrize("fmt", ["NV12", "I420", "BGRA"])
def test_chain_a_to_b_to_c_inside_one_batch(ctx, fmt):
    """src -> (stream 1) -> t1 -> (stream 2) -> t2 -> (stream 3) -> out, all queued before any
    launch, several times over so that a race would show."""
    ovs = _overlays(3, 900)
    for i, ov in enumerate(ovs):
        ctx.overlay_set_rectangles(700 + i, _rects(ov))
    ctx.set_batch(64, 0)
    try:
        frame = random_frame(fmt, W, H, 41)
        want = copy_planes(frame)
        for ov in ovs:
            want = oracle_blend(fmt, W, H, want, _rects(ov))
        bufs = [ctx.acquire(fmt, W, H) for _ in range(4)]
        bufs[0].upload(frame)
        for rep in range(5):
            before = ctx.stats()["launches"]
            t = None
            for i in range(3):
                t = ctx.submit(700 + i, fmt, W, H, bufs[i].c, bufs[i + 1].c)
            ctx.wait(t)
            assert ctx.stats()["launches"] - before == 3, "dependent frames must not share a launch"
            assert_planes_equal(bufs[3].download(), want, f"{fmt} chain, repetition {rep}")
        for b in bufs:
            b.release()
    finally:
        ctx.set_batch(32, 200)


def test_ping_pong_and_write_after_read(ctx):
    """A -> B then B -> A (the second frame overwrites what the first one reads), and a frame
    whose destination is another queued frame's source."""
    fmt = "NV12"
    ov1, ov2 = _overlays(2, 910)
    ctx.overlay_set_rectangles(710, _rects(ov1))
    ctx.overlay_set_rectangles(711, _rects(ov2))
    ctx.set_batch(64, 0)
    try:
        fa = random_frame(fmt, W, H, 42)
        a, b = ctx.acquire(fmt, W, H), ctx.acquire(fmt, W, H)
        a.upload(fa)
        want_b = oracle_blend(fmt, W, H, copy_planes(fa), _rects(ov1))
        want_a = oracle_blend(fmt, W, H, copy_planes(want_b), _rects(ov2))
        for rep in range(5):
            a.upload(fa)
            ctx.submit(710, fmt, W, H, a.c, b.c)
            ctx.wait(ctx.submit(711, fmt, W, H, b.c, a.c))
            assert_planes_equal(b.download(), want_b, f"ping, repetition {rep}")
            assert_planes_equal(a.download(), want_a, f"pong, repetition {rep}")
        # write after read: frame 2 writes into the buffer frame 1 reads from
        c = ctx.acquire(fmt, W, H)
        fc = random_frame(fmt, W, H, 43)
        for rep in range(5):
            a.upload(fa)
            c.upload(fc)
            ctx.submit(710, fmt, W, H, a.c, b.c)          # reads a
            ctx.wait(ctx.submit(711, fmt, W, H, c.c, a.c))  # writes a
            assert_planes_equal(b.download(), want_b, f"reader of a, repetition {rep}")
            assert_planes_equal(a.download(), oracle_blend(fmt, W, H, copy_planes(fc), _rects(ov2)),
                                f"writer of a, repetition {rep}")
        for f in (a, b, c):
            f.release()
    finally:
        ctx.set_batch(32, 200)


def test_shared_source_still_shares_a_launch(ctx):
    """Frames that only READ the same buffer do not depend on each other."""
    fmt = "NV12"
    ov = _overlays(1, 920)[0]
    ctx.overlay_set_rectangles(720, _rects(ov))
    ctx.set_batch(64, 0)
    try:
        src = ctx.acquire(fmt, W, H)
        frame = random_frame(fmt, W, H, 44)
        src.upload(frame)
        dsts = [ctx.acquire(fmt, W, H) for _ in range(6)]
        before = ctx.stats()["launches"]
        t = [ctx.submit(720, fmt, W, H, src.c, d.c) for d in dsts]
        ctx.wait(t[-1])
        assert ctx.stats()["launches"] - before == 1
        want = oracle_blend(fmt, W, H, copy_planes(frame), _rects(ov))
        for d in dsts:
            assert_planes_equal(d.download(), want, "shared source")
        for f in dsts + [src]:
            f.release()
    finally:
        ctx.set_batch(32, 200)


def test_overlapping_views_of_one_buffer_are_ordered(ctx):
    """The second frame's destination is a sub-view (other base pointer) of the first frame's
    destination: ranges are compared, not base pointers."""
    fmt = "GRAY8"
    ov_big = random_overlay(W, H, 930, density=0.6)
    ov_small = random_overlay(W // 2, H // 2, 931, density=0.6)
    ctx.overlay_set_rectangles(730, _rects(ov_big))
    ctx.overlay_set_rectangles(731, _rects(ov_small))
    ctx.set_batch(64, 0)
    try:
        big = ctx.acquire(fmt, W, H)
        frame = random_frame(fmt, W, H, 45)
        want = oracle_blend(fmt, W, H, copy_planes(frame), _rects(ov_big))
        x0, y0 = 160, 90                      # 16-byte aligned sub-view
        sub_want = [np.ascontiguousarray(want[0][y0:y0 + H // 2, x0:x0 + W // 2])]
        sub_want = oracle_blend(fmt, W // 2, H // 2, sub_want, _rects(ov_small))
        want[0][y0:y0 + H // 2, x0:x0 + W // 2] = sub_want[0]
        F = pkg.ttmlblend.Frame
        for rep in range(5):
            big.upload(frame)
            view = F()
            view.plane[0] = big.c.plane[0] + y0 * big.c.stride[0] + x0
            view.stride[0] = big.c.stride[0]
            ctx.submit(730, fmt, W, H, big.c, big.c)
            ctx.wait(ctx.submit(731, fmt, W // 2, H // 2, view, view))
            assert_planes_equal(big.download(), want, f"sub-view, repetition {rep}")
        big.release()
    finally:
        ctx.set_batch(32, 200)


@pytest.mark.parametrize("pinned", [True, False])
def test_two_overlays_on_one_host_frame(ctx, pinned):
    """Two streams' cues blended onto the same host frame back to back (zero copy when the frame
    is pinned, otherwise two staging jobs that must run one after the other)."""
    fmt = "NV12"
    ov1, ov2 = _overlays(2, 940)
    ctx.overlay_set_rectangles(740, _rects(ov1))
    ctx.overlay_set_rectangles(741, _rects(ov2))
    frame = random_frame(fmt, W, H, 46)
    want = oracle_blend(fmt, W, H, copy_planes(frame), _rects(ov1))
    want = oracle_blend(fmt, W, H, want, _rects(ov2))
    ctx.set_batch(64, 0)
    try:
        for rep in range(5):
            if pinned:
                hf = ctx.acquire(fmt, W, H, on_host=True)
                views = hf.host_planes()
                for v, p in zip(views, frame):
                    v[...] = p
                t1 = ctx.blend_host_frame(740, fmt, W, H, hf.c)
                t2 = ctx.blend_host_frame(741, fmt, W, H, hf.c)
                ctx.wait(t1)
                ctx.wait(t2)
                got = [v.copy() for v in views]
                hf.release()
            else:
                got = copy_planes(frame)
                t1 = ctx.blend_host(740, fmt, W, H, got)
                t2 = ctx.blend_host(741, fmt, W, H, got)
                ctx.wait(t1)
                ctx.wait(t2)
            assert_planes_equal(got, want, f"two overlays, pinned={pinned}, repetition {rep}")
    finally:
        ctx.set_batch(32, 200)


def test_host_forget_drops_automatic_registrations():
    """auto-register pins pageable frames on first sight; host_forget (what the owner calls before
    freeing the memory) unpins them again, and the next frame from such memory is staged or
    re-registered -- never blended through a stale mapping."""
    fmt = "NV12"
    c = pkg.TtmlBlend(0)
    try:
        ov = random_overlay(W, H, 950)
        c.overlay_set_rectangles(1, _rects(ov))
        c.set_auto_register(True)
        frame = random_frame(fmt, W, H, 47)
        want = oracle_blend(fmt, W, H, copy_planes(frame), _rects(ov))
        backing = np.empty(H * W * 2, dtype=np.uint8)        # both planes inside one allocation
        planes = [backing[:H * W].reshape(H, W), backing[H * W:H * W + (H // 2) * W].reshape(H // 2, W)]
        for rep in range(3):
            for p, s in zip(planes, frame):
                p[...] = s
            c.wait(c.blend_host(1, fmt, W, H, planes))
            assert_planes_equal(planes, want, f"auto-registered, repetition {rep}")
            assert c.host_forget(backing) >= 1
        assert c.host_forget(backing) == 0                   # nothing left
    finally:
        c.close()


@pytest.mark.parametrize("batch", [1, 3, 8])
@pytest.mark.parametrize("seed", range(4))
def test_random_dependency_chains(ctx, batch, seed):
    """Launches may overlap their predecessors (programmatic dependent launch) unless the range
    tracker finds a dependency: a random sequence of blends over a small pool of buffers --
    sources and destinations picked at random, in place now and then -- must give exactly what
    running them one after the other gives, whatever the batch size."""
    import random
    rnd = random.Random(9000 + seed)
    fmt, w, h = ("NV12", 320, 180) if seed % 2 == 0 else ("BGRA", 256, 144)
    ovs = [random_overlay(w, h, 960 + seed * 10 + i, density=0.5) for i in range(3)]
    for i, ov in enumerate(ovs):
        ctx.overlay_set_rectangles(760 + i, _rects(ov))
    ctx.set_batch(batch, 0)
    try:
        n_buf = 6
        bufs = [ctx.acquire(fmt, w, h) for _ in range(n_buf)]
        model = [random_frame(fmt, w, h, 50 + seed * 10 + i) for i in range(n_buf)]
        for b, m in zip(bufs, model):
            b.upload(m)
        before = ctx.stats()
        t = None
        for _ in range(80):
            s, d, k = rnd.randrange(n_buf), rnd.randrange(n_buf), rnd.randrange(3)
            if rnd.random() < 0.2:
                d = s
            t = ctx.submit(760 + k, fmt, w, h, bufs[s].c, bufs[d].c)
            model[d] = oracle_blend(fmt, w, h, copy_planes(model[s]), _rects(ovs[k]))
        ctx.flush()
        ctx.wait(t)
        after = ctx.stats()
        for i, (b, m) in enumerate(zip(bufs, model)):
            assert_planes_equal(b.download(), m, f"buffer {i} (batch {batch}, seed {seed})")
        if os.environ.get("FLUC_TTMLBLEND_PDL") != "0":
            assert after["dependent_launches"] > before["dependent_launches"]   # there were dependencies
        for b in bufs:
            b.release()
    finally:
        ctx.set_batch(32, 200)


def test_independent_launches_are_not_serialised(ctx):
    """Frames that share nothing with what is in flight are launched without waiting for it."""
    fmt = "NV12"
    ov = _overlays(1, 970)[0]
    ctx.overlay_set_rectangles(770, _rects(ov))
    ctx.set_batch(1, 0)
    try:
        srcs = [ctx.acquire(fmt, W, H) for _ in range(8)]
        dsts = [ctx.acquire(fmt, W, H) for _ in range(8)]
        frame = random_frame(fmt, W, H, 48)
        for s in srcs:
            s.upload(frame)
        ctx.sync()
        before = ctx.stats()
        t = [ctx.submit(770, fmt, W, H, s.c, d.c) for s, d in zip(srcs, dsts)]
        mid = ctx.stats()
        assert mid["launches"] - before["launches"] == 8
        assert mid["dependent_launches"] == before["dependent_launches"]
        # the same destinations again, nothing waited for: now a launch writes what one that may
        # still run writes
        t = [ctx.submit(770, fmt, W, H, s.c, d.c) for s, d in zip(srcs, dsts)]
        ctx.wait(t[-1])
        if os.environ.get("FLUC_TTMLBLEND_PDL") != "0":
            assert ctx.stats()["dependent_launches"] > mid["dependent_launches"]
        want = oracle_blend(fmt, W, H, copy_planes(frame), _rects(ov))
        for d in dsts:
            assert_planes_equal(d.download(), want, "independent launches")
        for f in srcs + dsts:
            f.release()
    finally:
        ctx.set_batch(32, 200)


def test_wait_for_a_retired_ticket_does_not_wait_for_the_batch_in_flight(ctx):
    """A caller that stays one batch behind waits for ticket i-1 after submitting batch i. When
    batch i-1 has already been retired, that wait is over at once -- it must not resolve to the next
    batch that is still in flight (it did: a C caller's pipeline then ran one batch at a time)."""
    import time
    fmt, w, h = "NV12", 1920, 1080
    ov = random_overlay(w, 120, 990, density=0.9)
    ctx.overlay_set_rectangles(790, [dict(pixels=ov, x=0, y=800)])
    n = 32
    ctx.set_batch(n, 0)
    try:
        srcs = [ctx.acquire(fmt, w, h) for _ in range(n)]
        dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
        frame = random_frame(fmt, w, h, 49)
        for s in srcs:
            s.upload(frame)
        ctx.sync()
        batch = ctx.Batch([790] * n, fmt, w, h, [s.c for s in srcs], [d.c for d in dsts])
        best = None
        for attempt in range(3):
            old = ctx.submit_many(batch)[n - 1]
            ctx.flush()
            ctx.wait(old)                               # finished and retired
            ctx.submit_many_repeat(batch, 400)          # 12800 frames in flight: tens of ms
            newest = ctx.submit_many(batch)[n - 1]
            ctx.flush()
            t0 = time.perf_counter()
            ctx.wait(old)
            t1 = time.perf_counter()
            ctx.wait(newest)
            t2 = time.perf_counter()
            ratio = (t1 - t0) / max(t2 - t0, 1e-9)
            best = ratio if best is None else min(best, ratio)
            if best < 0.1:
                break
        assert best < 0.1, f"wait (retired ticket) took {best:.2f} of the time the work in flight needed"
        want = oracle_blend(fmt, w, h, copy_planes(frame), [dict(pixels=ov, x=0, y=800)])
        assert_planes_equal(dsts[n - 1].download(), want, "after the waits")
        for f in srcs + dsts:
            f.release()
    finally:
        ctx.set_batch(32, 200)


def test_host_dma_batches(ctx):
    """Pinned pool frames come in slabs (constant spacing), so a batch of them can be moved by the
    copy engines -- one 2-D copy per piece of rows and run of frames -- blended in device staging and
    copied back (fluc_ttmlblend_set_host_dma; zero copy otherwise). Same bytes as the oracle either
    way; a second batch on the same frames waits for the first one, and so does a single zero-copy
    frame. Repetition 0 runs with the context's default (the transport is chosen by measurement unless
    the environment says otherwise), 1 and 2 with the copy engines."""
    fmt, W, H = "NV12", 1024, 360          # 1024: pool stride == row bytes, the windows are whole rows
    box = lambda seed: np.ascontiguousarray(np.concatenate(
        [np.zeros((200, W, 4), np.uint8), _opaque_free(random_overlay(W, 120, seed, density=0.9)), np.zeros((40, W, 4), np.uint8)]))
    ov1, ov2 = box(980), box(981)
    ctx.overlay_set(780, ov1, [(0, 200, W, 120)])
    ctx.overlay_set(781, ov2, [(0, 200, W, 120)])
    n = 16
    ctx.set_batch(n, 0)
    try:
        hosts = [ctx.acquire(fmt, W, H, on_host=True) for _ in range(n)]
        frames = [random_frame(fmt, W, H, 70 + i) for i in range(n)]
        for rep in range(3):
            if rep == 1:
                ctx.set_host_dma(1)
            for hf, fr in zip(hosts, frames):
                for v, p in zip(hf.host_planes(), fr):
                    v[...] = p
            before = ctx.stats()
            b1 = ctx.Batch([780] * n, fmt, W, H, [h.c for h in hosts], [h.c for h in hosts])
            b2 = ctx.Batch([781] * n, fmt, W, H, [h.c for h in hosts], [h.c for h in hosts])
            t1 = ctx.blend_host_many(b1)
            t2 = ctx.blend_host_many(b2)                            # the same frames again, nothing waited for
            t3 = ctx.blend_host_frame(780, fmt, W, H, hosts[3].c)   # and one of them once more, zero copy
            ctx.flush()
            ctx.wait(t1[n - 1])
            ctx.wait(t2[n - 1])
            ctx.wait(t3)
            after = ctx.stats()
            if (rep >= 1 or os.environ.get("FLUC_TTMLBLEND_HOST_DMA") == "1") \
                    and "FLUC_TTMLBLEND_GROUPS" not in os.environ and "FLUC_TTMLBLEND_LAZY" not in os.environ:
                assert after["host_dma_batches"] - before["host_dma_batches"] >= 2, after     # in pieces of 8 frames
            for i, (hf, fr) in enumerate(zip(hosts, frames)):
                want = oracle_blend(fmt, W, H, copy_planes(fr), _rects(ov1))
                want = oracle_blend(fmt, W, H, want, _rects(ov2))
                if i == 3:
                    want = oracle_blend(fmt, W, H, want, _rects(ov1))
                assert_planes_equal([v.copy() for v in hf.host_planes()], want, f"host frame {i}, repetition {rep}")
        for h in hosts:
            h.release()
    finally:
        ctx.set_host_dma(int(os.environ.get("FLUC_TTMLBLEND_HOST_DMA", "2")))
        ctx.set_batch(32, 200)


def _opaque_free(img):
    """A translucent cue (no opaque vectors: such batches take the copy engines)."""
    img = img.copy()
    a = img[..., 3].astype(np.uint32)
    a = np.minimum(a, 200)
    a[a == 0] = 120                                   # a translucent box behind everything
    img[..., 3] = a
    img[..., :3] = np.minimum(img[..., :3], img[..., 3:4])      # stays valid premultiplied data
    return img
