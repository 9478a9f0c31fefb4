"""Frames that other CUDA streams produce and consume: fluc_ttmlblend_submit_many_after orders the
blend after the work already enqueued on the caller's stream, fluc_ttmlblend_wait_on_stream lets a
stream wait for the blend, and the host blocks in neither. torch is only the plumbing here:
producer streams held back by torch.cuda._sleep, frames written and read with copy_. Every result
is compared with the oracle's sequential blend, tolerance 0, after one torch.cuda.synchronize().

Every held run is done twice (REPS). The first launch of a kernel in a process loads it (CUDA's
lazy module loading), which may synchronise the context: with the stream waits removed, such first
runs still came out right, so only the later ones check the waits."""
import ctypes
import random

import numpy as np
import pytest
import torch

from helpers import assert_planes_equal, copy_planes, oracle_blend, pkg, random_frame, random_overlay

pytestmark = pytest.mark.gpu

tb = pkg.ttmlblend
W, H = 640, 360
SLEEP = 100_000_000          # GPU clock cycles: about 50 ms on a B200
REPS = 2


def _rects(ov):
    return [dict(pixels=ov, x=0, y=0)]


def _dev(planes):
    """Device copies of numpy planes, one contiguous uint8 tensor per plane."""
    return [torch.from_numpy(np.ascontiguousarray(p)).cuda() for p in planes]


def _frame(tensors):
    f = tb.Frame()
    for i, t in enumerate(tensors):
        f.plane[i] = t.data_ptr()
        f.stride[i] = t.stride(0)
    return f


def _host(tensors):
    return [t.cpu().numpy() for t in tensors]


def _batch(ctx, stream, fmt, w, h, srcs, dsts):
    return ctx.Batch([stream] * len(srcs), fmt, w, h, [_frame(s) for s in srcs], [_frame(d) for d in dsts])


@pytest.fixture
def cue(ctx):
    """Library stream 850 with a cue over the whole 640x360 frame; batch settings restored."""
    ov = random_overlay(W, H, 1850, density=0.6)
    ctx.overlay_set_rectangles(850, _rects(ov))
    yield 850, _rects(ov)
    ctx.set_batch(32, 200)


def _held_producer(srcs, news):
    """A stream that sleeps, then writes `news` into `srcs`: frames a decoder is still producing."""
    p = torch.cuda.Stream()
    with torch.cuda.stream(p):
        torch.cuda._sleep(SLEEP)
        for s, n in zip(srcs, news):
            for a, b in zip(s, n):
                a.copy_(b)
    return p


@pytest.mark.parametrize("inplace", [False, True], ids=["out", "inplace"])
@pytest.mark.parametrize("fmt", ["NV12", "I420", "BGRA"])
def test_blend_reads_what_the_producer_wrote(ctx, cue, fmt, inplace):
    """The frames hold X; the producer stream sleeps, then writes Y. A blend submitted after that
    stream gives blend(Y), never blend(X)."""
    stream, rects = cue
    for rep in range(REPS):
        x, y = random_frame(fmt, W, H, 1 + 2 * rep), random_frame(fmt, W, H, 2 + 2 * rep)
        src, ynew = _dev(x), _dev(y)
        dst = src if inplace else [torch.zeros_like(t) for t in src]
        torch.cuda.synchronize()
        p = _held_producer([src], [ynew])
        t = ctx.submit_many_after(_batch(ctx, stream, fmt, W, H, [src], [dst]), p.cuda_stream)[0]
        ctx.wait(t)
        torch.cuda.synchronize()
        assert_planes_equal(_host(dst), oracle_blend(fmt, W, H, copy_planes(y), rects),
                            f"{fmt} inplace={inplace}, repetition {rep}")


def _held_blend_and_consumer(ctx, stream, fmt, seed):
    """A blend held behind a sleeping producer, and a consumer stream that waits for it and then
    copies the destination out. Returns the producer and consumer streams, the copy, the planes the
    producer wrote, and the buffers, which must outlive the streams' work."""
    x, y = random_frame(fmt, W, H, seed), random_frame(fmt, W, H, seed + 1)
    src, ynew = _dev(x), _dev(y)
    dst = [torch.zeros_like(t) for t in src]
    out = [torch.zeros_like(t) for t in src]
    torch.cuda.synchronize()
    p = _held_producer([src], [ynew])
    t = ctx.submit_many_after(_batch(ctx, stream, fmt, W, H, [src], [dst]), p.cuda_stream)[0]
    s2 = torch.cuda.Stream()
    ctx.wait_on_stream(t, s2.cuda_stream)
    with torch.cuda.stream(s2):
        for o, d in zip(out, dst):
            o.copy_(d)
    return p, s2, out, y, (src, ynew, dst)


def test_consumer_stream_waits_for_the_blend(ctx, cue):
    stream, rects = cue
    for rep in range(REPS):
        _, _, out, y, keep = _held_blend_and_consumer(ctx, stream, "NV12", 10 + 2 * rep)
        torch.cuda.synchronize()
        assert_planes_equal(_host(out), oracle_blend("NV12", W, H, copy_planes(y), rects),
                            f"consumer copy, repetition {rep}")


def test_the_host_does_not_block(ctx, cue):
    """Both calls have returned while the producer is still asleep: neither waited for the GPU
    (checked on the last repetition, once the kernels are loaded)."""
    stream, _ = cue
    for rep in range(REPS):
        p, s2, _, _, keep = _held_blend_and_consumer(ctx, stream, "NV12", 20 + 2 * rep)
        asleep = not p.query(), not s2.query()
        torch.cuda.synchronize()
    assert asleep == (True, True)


def test_ticket_cases(ctx, cue):
    stream, rects = cue
    lib = ctx.lib
    s2 = torch.cuda.Stream()
    x = random_frame("NV12", W, H, 5)
    src = _dev(x)
    dst = [torch.zeros_like(t) for t in src]
    torch.cuda.synchronize()
    ctx.set_batch(32, 0)                                 # only wait / flush / the limit launch
    b = _batch(ctx, stream, "NV12", W, H, [src], [dst])
    t = ctx.submit_many_after(b, s2.cuda_stream)[0]
    before = ctx.stats()["launches"]
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, t, s2.cuda_stream) == tb.OK
    assert ctx.stats()["launches"] > before, "a queued ticket is launched"
    ctx.wait(t)
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, t, s2.cuda_stream) == tb.OK       # retired
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, t, None) == tb.OK                 # legacy default stream
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, 0, s2.cuda_stream) == tb.ERROR_NOT_FOUND
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, t + 1000, s2.cuda_stream) == tb.ERROR_NOT_FOUND
    assert lib.fluc_ttmlblend_wait_on_stream(None, t, s2.cuda_stream) == tb.ERROR_INVALID_ARGUMENT
    tickets = (ctypes.c_uint64 * 1)()
    assert lib.fluc_ttmlblend_submit_many_after(None, s2.cuda_stream, b.n, b.streams, b.fmt, b.width, b.height,
                                                b.flags, b.srcs, b.dsts, tickets) == tb.ERROR_INVALID_ARGUMENT
    # a zero-copy host frame: its batch's event covers it
    hf = ctx.acquire("NV12", W, H, on_host=True)
    views = hf.host_planes()
    for v, p in zip(views, x):
        v[...] = p
    th = ctx.blend_host_frame(stream, "NV12", W, H, hf.c)
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, th, s2.cuda_stream) == tb.OK
    # a staged host frame (pageable, not 16-byte aligned) ends with a CPU copy
    backing = [np.zeros((r, c + 17), np.uint8) for r, c in ((H, W), (H // 2, W))]
    planes = [bk[:, 1:1 + p.shape[1]] for bk, p in zip(backing, x)]
    for dv, p in zip(planes, x):
        dv[...] = p
    staged = ctx.stats()["staged_frames"]
    ts = ctx.blend_host(stream, "NV12", W, H, planes)
    assert ctx.stats()["staged_frames"] == staged + 1
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, ts, s2.cuda_stream) == tb.ERROR_INVALID_ARGUMENT
    ctx.wait(ts)
    torch.cuda.synchronize()
    want = oracle_blend("NV12", W, H, copy_planes(x), rects)
    assert_planes_equal(_host(dst), want, "device frame")
    assert_planes_equal([v.copy() for v in views], want, "zero-copy host frame")
    assert_planes_equal(planes, want, "staged host frame")
    hf.release()


def test_stream_of_another_device_is_rejected(ctx, cue):
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    stream, _ = cue
    src = _dev(random_frame("NV12", W, H, 6))
    torch.cuda.synchronize()
    b = _batch(ctx, stream, "NV12", W, H, [src], [src])
    with torch.cuda.device(1):
        other = torch.cuda.Stream()
    tickets = (ctypes.c_uint64 * 1)()
    lib = ctx.lib
    assert lib.fluc_ttmlblend_submit_many_after(ctx.h, other.cuda_stream, b.n, b.streams, b.fmt, b.width,
                                                b.height, b.flags, b.srcs, b.dsts, tickets) == tb.ERROR_INVALID_ARGUMENT
    t = ctx.submit(stream, "NV12", W, H, b.srcs[0], b.dsts[0])
    assert lib.fluc_ttmlblend_wait_on_stream(ctx.h, t, other.cuda_stream) == tb.ERROR_INVALID_ARGUMENT
    ctx.wait(t)


def test_many_producers_share_a_launch(ctx):
    """8 producer streams with different sleep lengths, one call each, default linger: the frames
    share launches, and every one of them is blended from what its own producer wrote."""
    ov = random_overlay(W, H, 1860, density=0.6)
    for i in range(8):
        ctx.overlay_set_rectangles(860 + i, _rects(ov))
    ctx.set_batch(32, 200)
    for rep in range(REPS):
        xs = [random_frame("NV12", W, H, 100 + 20 * rep + i) for i in range(8)]
        ys = [random_frame("NV12", W, H, 110 + 20 * rep + i) for i in range(8)]
        srcs, news = [_dev(x) for x in xs], [_dev(y) for y in ys]
        dsts = [[torch.zeros_like(t) for t in s] for s in srcs]
        batches = [_batch(ctx, 860 + i, "NV12", W, H, [srcs[i]], [dsts[i]]) for i in range(8)]
        torch.cuda.synchronize()
        producers = []
        for i in range(8):
            p = torch.cuda.Stream()
            with torch.cuda.stream(p):
                torch.cuda._sleep(SLEEP // 16 * (i + 1))
                for a, b in zip(srcs[i], news[i]):
                    a.copy_(b)
            producers.append(p)
        before = ctx.stats()["launches"]
        tickets = [ctx.submit_many_after(b, p.cuda_stream)[0] for b, p in zip(batches, producers)]
        for t in tickets:
            ctx.wait(t)
        launches = ctx.stats()["launches"] - before
        assert launches < 8, f"{launches} launches for 8 one-frame calls, repetition {rep}"
        torch.cuda.synchronize()
        for i in range(8):
            assert_planes_equal(_host(dsts[i]), oracle_blend("NV12", W, H, copy_planes(ys[i]), _rects(ov)),
                                f"producer {i}, repetition {rep}")


def test_one_call_over_several_launches(ctx, cue):
    """13 frames at 4 per launch: waiting on the stream for the last ticket covers all of them."""
    stream, rects = cue
    w, h, n = 320, 180, 13
    ov = random_overlay(w, h, 1870, density=0.6)
    ctx.overlay_set_rectangles(stream, _rects(ov))
    ctx.set_batch(4, 0)
    for rep in range(REPS):
        xs = [random_frame("NV12", w, h, 200 + 40 * rep + i) for i in range(n)]
        ys = [random_frame("NV12", w, h, 220 + 40 * rep + i) for i in range(n)]
        srcs, news = [_dev(x) for x in xs], [_dev(y) for y in ys]
        dsts = [[torch.zeros_like(t) for t in s] for s in srcs]
        outs = [[torch.zeros_like(t) for t in s] for s in srcs]
        torch.cuda.synchronize()
        p = _held_producer(srcs, news)
        before = ctx.stats()["launches"]
        tickets = ctx.submit_many_after(_batch(ctx, stream, "NV12", w, h, srcs, dsts), p.cuda_stream)
        s2 = torch.cuda.Stream()
        ctx.wait_on_stream(tickets[n - 1], s2.cuda_stream)
        assert ctx.stats()["launches"] - before >= 4
        with torch.cuda.stream(s2):
            for o, d in zip(outs, dsts):
                for a, b in zip(o, d):
                    a.copy_(b)
        torch.cuda.synchronize()
        for i in range(n):
            assert_planes_equal(_host(outs[i]), oracle_blend("NV12", w, h, copy_planes(ys[i]), _rects(ov)),
                                f"frame {i}, repetition {rep}")


def test_mixed_callers_in_one_launch(ctx, cue):
    """submit_many frames whose sources are ready and submit_many_after frames whose producer is
    still asleep, in one launch: that launch waits for the producer, and every frame is right."""
    stream, rects = cue
    ctx.set_batch(32, 0)
    for rep in range(REPS):
        xs = [random_frame("NV12", W, H, 300 + 10 * rep + i) for i in range(6)]
        y = [random_frame("NV12", W, H, 306 + 10 * rep + i) for i in range(3)]
        srcs = [_dev(x) for x in xs]
        dsts = [[torch.zeros_like(t) for t in s] for s in srcs]
        news = [_dev(v) for v in y]
        torch.cuda.synchronize()
        p = _held_producer(srcs[3:], news)
        before = ctx.stats()["launches"]
        ctx.submit_many(_batch(ctx, stream, "NV12", W, H, srcs[:3], dsts[:3]))
        t = ctx.submit_many_after(_batch(ctx, stream, "NV12", W, H, srcs[3:], dsts[3:]), p.cuda_stream)[2]
        ctx.wait(t)
        assert ctx.stats()["launches"] - before == 1
        torch.cuda.synchronize()
        for i, base in enumerate(xs[:3] + y):
            assert_planes_equal(_host(dsts[i]), oracle_blend("NV12", W, H, copy_planes(base), rects),
                                f"frame {i}, repetition {rep}")


def test_chain_across_streams(ctx):
    """A is blended after its producer; stream S2 waits for A, rewrites part of it and submits it,
    after S2, as the source of B. Both equal the sequential composition."""
    ov1, ov2 = random_overlay(W, H, 1880, density=0.5), random_overlay(W, H, 1881, density=0.5)
    ctx.overlay_set_rectangles(880, _rects(ov1))
    ctx.overlay_set_rectangles(881, _rects(ov2))
    for rep in range(REPS):
        x, y = random_frame("NV12", W, H, 400 + 2 * rep), random_frame("NV12", W, H, 401 + 2 * rep)
        src, ynew = _dev(x), _dev(y)
        a = [torch.zeros_like(t) for t in src]
        b = [torch.zeros_like(t) for t in src]
        torch.cuda.synchronize()
        p = _held_producer([src], [ynew])
        ta = ctx.submit_many_after(_batch(ctx, 880, "NV12", W, H, [src], [a]), p.cuda_stream)[0]
        s2 = torch.cuda.Stream()
        ctx.wait_on_stream(ta, s2.cuda_stream)
        with torch.cuda.stream(s2):
            torch.cuda._sleep(SLEEP // 4)
            a[0][100:140].fill_(77)
        t_b = ctx.submit_many_after(_batch(ctx, 881, "NV12", W, H, [a], [b]), s2.cuda_stream)[0]
        ctx.wait(t_b)
        torch.cuda.synchronize()
        want_a = oracle_blend("NV12", W, H, copy_planes(y), _rects(ov1))
        want_a[0][100:140] = 77
        assert_planes_equal(_host(a), want_a, f"A, rewritten by S2, repetition {rep}")
        assert_planes_equal(_host(b), oracle_blend("NV12", W, H, copy_planes(want_a), _rects(ov2)),
                            f"B, repetition {rep}")


@pytest.mark.parametrize("batch", [1, 3, 8])
@pytest.mark.parametrize("seed", range(2))
def test_random_stream_chains(ctx, batch, seed):
    """A random sequence over a small pool of buffers: blends submitted after one of three CUDA
    streams, and edits on those streams, each edit made after waiting on its stream for every blend
    that touched the buffer. The result equals running the sequence one step after the other."""
    rnd = random.Random(9100 + seed)
    fmt, w, h = ("NV12", 320, 180) if seed % 2 == 0 else ("BGRA", 256, 144)
    ovs = [random_overlay(w, h, 1890 + seed * 10 + i, density=0.5) for i in range(3)]
    for i, ov in enumerate(ovs):
        ctx.overlay_set_rectangles(890 + i, _rects(ov))
    ctx.set_batch(batch, 0)
    try:
        n_buf = 6
        model = [random_frame(fmt, w, h, 100 + seed * 10 + i) for i in range(n_buf)]
        bufs = [_dev(m) for m in model]
        streams = [torch.cuda.Stream() for _ in range(3)]
        last_ticket = [0] * n_buf           # newest blend that read or wrote the buffer
        editor = [None] * n_buf             # stream of the newest edit of the buffer
        torch.cuda.synchronize()
        for _ in range(60):
            s = rnd.randrange(3)
            st = streams[s]
            if rnd.random() < 0.3:
                # edit: after every blend that touched it, and after its previous edit
                d = rnd.randrange(n_buf)
                if last_ticket[d]:
                    ctx.wait_on_stream(last_ticket[d], st.cuda_stream)
                if editor[d] is not None and editor[d] is not st:
                    st.wait_stream(editor[d])
                r0 = rnd.randrange(h - 8)
                val = rnd.randrange(256)
                with torch.cuda.stream(st):
                    if rnd.random() < 0.5:
                        torch.cuda._sleep(SLEEP // 50)
                    bufs[d][0][r0:r0 + 8].fill_(val)
                model[d][0][r0:r0 + 8] = val
                editor[d] = st
            else:
                sb, d, k = rnd.randrange(n_buf), rnd.randrange(n_buf), rnd.randrange(3)
                if rnd.random() < 0.2:
                    d = sb
                for e in {editor[sb], editor[d]}:
                    if e is not None and e is not st:
                        st.wait_stream(e)
                t = ctx.submit_many_after(_batch(ctx, 890 + k, fmt, w, h, [bufs[sb]], [bufs[d]]), st.cuda_stream)[0]
                last_ticket[sb] = last_ticket[d] = t
                model[d] = oracle_blend(fmt, w, h, copy_planes(model[sb]), _rects(ovs[k]))
        ctx.flush()
        torch.cuda.synchronize()
        for i, (b, m) in enumerate(zip(bufs, model)):
            assert_planes_equal(_host(b), m, f"buffer {i} (batch {batch}, seed {seed})")
    finally:
        ctx.set_batch(32, 200)
