"""Frames above 4K, up to the 32768-pixel limit of check_frame. Above 4K the host cuts work in ways
a 4K frame never reaches, and this file runs each of them on the GPU against `helpers.model_blend`
at tolerance 0 (out of place the rest of the frame equals the source, in place it is untouched):

A. 8K UHD (7680 x 4320) in RGBA, BGRA, AYUV, ARGB, RGB, v308, NV12 and I420: a full-width
   rectangle tall enough that push_window cuts its window into pieces (1344 rows a piece for the
   packed kinds, 2519 for the 3-byte kinds; NV12 and I420 are not cut and are the control), a
   narrower one sharing some of its rows (a JC_GENERAL window), a sparse cue (lazy in place) or one
   with an opaque box (opaque skip out of place); out of place, in place, pinned host frames (zero
   copy), pageable host frames (staged), on pool frames and on frames with a padded stride; a
   rectangle hanging off the right and bottom edges; a batch of pinned frames through the copy
   engines (host DMA) whose windows are cut into pieces;
B. geometries whose group launch would not be exact for a full group of frames (make_groupable),
   so their fast windows go to the table kernel: 8192 x 4320 RGBA and Y444, 7680 x 4320 RGB, each
   as a batch of four frames sharing the cue;
C. near the limit: 32764 x 1024 BGRA and AYUV (64-row pieces; BGRA in place takes the table
   kernel), 32767-wide GRAY8 and I420 (a ragged last vector column for the byte kernel next to the
   group launch), 15360 x 8640 RGBA (312-row pieces, table kernel out of place);
D. byte offsets past 2^31 and 2^32: 256-wide GRAY8 and NV12 frames of 32768 rows with strides of
   2^17 + 256 (group kernel) and 2^17 + 259 (byte kernel), rectangles at the top, across row 16384
   and on rows that start beyond 2^32; one 32768 x 32768 BGRA frame under a frame-sized cue whose
   prepared plane is 4 GiB, checked on sampled rows. An offset narrowed to 32 bits would address
   the wrong bytes here, so these cases cover that class of bug by construction;
E. a move at 8K: the tall rectangle of A shifted by an odd number of rows and columns, so that the
   piece boundaries fall elsewhere; against the model and a fresh install.

Which path a case takes (pieces, group or table kernel, lazy, opaque skip, host DMA) is asserted only
when no FLUC_TTMLBLEND_* knob is set: under a knob every comparison still runs. The cases use a
context of their own, closed at the end of the module, so that the frames its pool keeps do not stay
allocated for the rest of the run; frames with odd strides and the frames above 2 GiB are torch
buffers, freed before the next test."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import test_host_logic as hl
from helpers import assert_planes_equal, copy_planes, model_blend, pkg, random_frame, random_overlay

pytestmark = pytest.mark.gpu

tb = pkg.ttmlblend
KNOB = any(k.startswith("FLUC_TTMLBLEND_") and k != "FLUC_TTMLBLEND_LIB" for k in os.environ)
W8, H8 = 7680, 4320
RGB24 = ("RGB", "v308")
_peak = [0]


def note_mem():
    """Device memory in use by this process and everything else on the GPU, for the peak."""
    free, total = torch.cuda.mem_get_info()
    _peak[0] = max(_peak[0], total - free)


@pytest.fixture(scope="module")
def gctx(lib):
    torch.cuda.init()
    free0, total = torch.cuda.mem_get_info()
    c = pkg.TtmlBlend(0)
    yield c
    c.close()
    torch.cuda.empty_cache()
    print(f"\ntest_gpu_geometry: peak device memory in use {(_peak[0] - (total - free0)) / 2**30:.2f} GiB "
          f"above the {(total - free0) / 2**30:.2f} GiB in use before the module")


@pytest.fixture(scope="module")
def hooks():
    return hl.load_hooks()


max_rows = hl.max_rows_of


def layout_jobs(hooks, fmt, w, h, rects, windowed):
    """The jobs the host builds for this frame and these (x, y, w, h) rectangles (CPU hook)."""
    return hl.build(hooks, fmt, w, h, hl.plane_rects(fmt, w, h, rects), windowed=windowed)[0]


def split(jobs):
    return any(j.win_rows == max_rows(j.win_nv) and j.win_nv > 1 for j in jobs)


# ---------------------------------------------------------------------------------------------
# frames

class TorchFrame:
    """All planes of a frame in one torch device buffer, each plane with stride row bytes + pad
    (or the strides given); bytes outside the rows start as `fill`."""

    def __init__(self, fmt, w, h, pad=0, strides=None, fill=0x5A):
        self.fmt, self.w, self.h = fmt, w, h
        self.layout = tb.plane_layout(fmt, w, h)
        self.strides = strides or [rb + pad for rb, _ in self.layout]
        total = sum(s * rows for s, (_, rows) in zip(self.strides, self.layout))
        self.buf = torch.full((total,), fill, dtype=torch.uint8, device="cuda")
        self.planes, off = [], 0
        self.c = tb.Frame()
        for i, (s, (rb, rows)) in enumerate(zip(self.strides, self.layout)):
            t = self.buf[off:off + s * rows].view(rows, s)
            self.planes.append(t)
            self.c.plane[i] = t.data_ptr()
            self.c.stride[i] = s
            off += s * rows

    def views(self):
        return [t[:, :rb] for t, (rb, _) in zip(self.planes, self.layout)]

    def upload(self, planes):
        for v, p in zip(self.views(), planes):
            v.copy_(torch.from_numpy(np.ascontiguousarray(p)))

    def download(self):
        return [v.cpu().numpy() for v in self.views()]

    def padding_is(self, fill):
        return all(bool((t[:, rb:] == fill).all()) for t, (rb, _) in zip(self.planes, self.layout))


def padded_host(planes, pad):
    """Pageable host planes with stride row bytes + pad."""
    out = []
    for p in planes:
        buf = np.full((p.shape[0], p.shape[1] + pad), 0x5A, np.uint8)
        buf[:, :p.shape[1]] = p
        out.append(buf[:, :p.shape[1]])
    return out


def blend(ctx, stream, fmt, w, h, frame, mode, pad=0):
    """One frame through the stream's overlay. mode: out / inplace (pool frames, or torch frames
    with a padded stride when pad > 0), zerocopy (pinned pool frame), staged (pageable)."""
    if mode == "staged":
        out = padded_host(frame, pad) if pad else copy_planes(frame)
        ctx.wait(ctx.blend_host(stream, fmt, w, h, out))
        return out
    if mode == "zerocopy":
        p = ctx.acquire(fmt, w, h, on_host=True)
        try:
            for d, s in zip(p.host_planes(), frame):
                d[...] = s
            ctx.wait(ctx.blend_host_frame(stream, fmt, w, h, p.c))
            return [np.array(x) for x in p.host_planes()]
        finally:
            p.release()
    if pad:
        src = TorchFrame(fmt, w, h, pad)
        src.upload(frame)
        dst = src if mode == "inplace" else TorchFrame(fmt, w, h, pad, fill=0xA5)
        note_mem()
        torch.cuda.synchronize()        # torch's copies are done before the library reads the frame
        ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dst.c))
        assert dst.padding_is(0x5A if mode == "inplace" else 0xA5), "bytes past the row written"
        return dst.download()
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


def delta(ctx, before):
    now = ctx.stats()
    return {k: now[k] - before[k] for k in before}


def clear_and_check(ctx, streams, base):
    """Clear the streams' overlays: the cache goes back to where it was."""
    for s in streams:
        ctx.overlay_clear(s)
    ctx.sync()
    ctx.sync()
    torch.cuda.empty_cache()
    assert ctx.stats()["cache_bytes"] == base


# ---------------------------------------------------------------------------------------------
# cues

_ov = {}


def overlay(kind, w, h):
    """kind: sparse (half of the 16-pixel groups transparent: lazy in place), box (an opaque box
    over most of the rectangle: opaque skip out of place), plain, translucent (no transparent and
    no opaque groups: neither). The first and last columns keep some alpha in every row, so that
    the row-span crop keeps the rectangle as it is."""
    key = (kind, w, h)
    if key in _ov:
        return _ov[key]
    img = random_overlay(w, h, 1000 + 7 * len(kind) + w % 97 + h % 89)
    if kind == "sparse":
        y, x = np.mgrid[0:h, 0:w]
        off = ((x // 16 + y // 4) % 2 == 0) & (x >= 16) & (x < w - 16)
        img[off] = 0
    elif kind == "box":
        img[h // 8:h - h // 8, w // 8:w - w // 8, 3] = 255
    elif kind == "translucent":
        a = img[..., 3]
        a[a == 0] = 120
        np.minimum(a, 200, out=a)
        np.minimum(img[..., :3], a[..., None], out=img[..., :3])
    img[:, 0, 3] = np.maximum(img[:, 0, 3], 1)
    img[:, -1, 3] = np.maximum(img[:, -1, 3], 1)
    _ov[key] = img
    return img


def cue_8k(fmt, kind):
    """A: the full-width rectangle (1500 rows, 2700 for the 3-byte kinds) and a narrower one over
    its last 100 rows and 500 rows below; the band where the tall one is alone is longer than a
    piece. Both end above the bottom edge."""
    tall = 2700 if fmt in RGB24 else 1500
    big = overlay(kind, W8, 2700)[:tall]
    return [dict(pixels=big, x=0, y=200),
            dict(pixels=overlay("plain", 1200, 600), x=2000, y=200 + tall - 100)]


def boxes(rl):
    return [(r["x"], r["y"], r["pixels"].shape[1], r["pixels"].shape[0]) for r in rl]


# ---------------------------------------------------------------------------------------------
# A. 8K UHD

A_CASES = [("RGBA", "sparse"), ("BGRA", "box"), ("AYUV", "sparse"), ("ARGB", "box"),
           ("RGB", "sparse"), ("v308", "box"), ("NV12", "sparse"), ("I420", "box")]
# out of place and staged host frames / in place and pinned host frames, each on pool frames and
# on frames with a padded stride. The two halves of a format run one after the other and share
# the model.
MODES = {"out": (("out", 0), ("staged", 0), ("out", 256), ("staged", 256)),
         "inplace": (("inplace", 0), ("zerocopy", 0), ("inplace", 256))}
_model = {}


def model_8k(fmt, kind, seed):
    key = (fmt, kind, seed)
    if key not in _model:
        _model.clear()
        frame = random_frame(fmt, W8, H8, seed)
        rl = cue_8k(fmt, kind)
        _model[key] = (frame, rl, model_blend(fmt, W8, H8, copy_planes(frame), rl))
    return _model[key]


@pytest.mark.parametrize("fmt,kind,place", [(f, k, p) for f, k in A_CASES for p in MODES])
def test_8k_split_windows(gctx, hooks, fmt, kind, place):
    ctx, st = gctx, 4000 + A_CASES.index((fmt, kind))
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    frame, rl, want = model_8k(fmt, kind, 11)
    ctx.overlay_set_rectangles(st, rl)
    jobs = {m: layout_jobs(hooks, fmt, W8, H8, boxes(rl), m == "inplace") for m in ("out", "inplace")}
    if not KNOB:
        for m in jobs:
            assert split(jobs[m]) == (fmt not in ("NV12", "I420")), m
    ctx.set_host_dma(0)
    try:
        for mode, pad in MODES[place]:
            s0 = ctx.stats()
            got = blend(ctx, st, fmt, W8, H8, frame, mode, pad)
            d = delta(ctx, s0)
            assert_planes_equal(got, want, f"{fmt} {kind} {mode} pad {pad}")
            if not KNOB and mode in ("out", "inplace"):
                # out of place the 3-byte kinds fall back to the table kernel (make_groupable)
                grouped = any(j.grouped for j in jobs[mode])
                assert (d["group_launches"] + d["multi_launches"] >= 1) == grouped, (mode, d)
                assert grouped == (mode == "inplace" or fmt not in RGB24)
                if grouped and kind == "sparse" and mode == "inplace":
                    assert d["lazy_launches"] >= 1, d
                if grouped and kind == "box" and mode == "out":
                    assert d["opaque_skip_launches"] >= 1, d
    finally:
        ctx.set_host_dma(int(os.environ.get("FLUC_TTMLBLEND_HOST_DMA", "2")))
    clear_and_check(ctx, [st], base)


@pytest.mark.parametrize("fmt", ["BGRA", "NV12"])
def test_8k_rectangle_over_the_right_and_bottom_edges(gctx, hooks, fmt):
    ctx, st = gctx, 4010 + ["BGRA", "NV12"].index(fmt)
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    frame = random_frame(fmt, W8, H8, 12)
    rl = [dict(pixels=overlay("plain", 7600, 1600), x=300, y=H8 - 1500)]
    want = model_blend(fmt, W8, H8, copy_planes(frame), rl)
    ctx.overlay_set_rectangles(st, rl)
    if not KNOB and fmt == "BGRA":
        assert split(layout_jobs(hooks, fmt, W8, H8, boxes(rl), False))
    for mode, pad in (("out", 0), ("inplace", 0), ("staged", 0), ("out", 256), ("inplace", 256)):
        assert_planes_equal(blend(ctx, st, fmt, W8, H8, frame, mode, pad), want, f"{fmt} {mode} pad {pad}")
    clear_and_check(ctx, [st], base)


def test_8k_host_dma_batch_of_split_windows(gctx, hooks):
    """Four pinned BGRA frames in place through the copy engines: the rows under the full-width
    rectangle go to device staging in one 2-D copy per run, are blended there in pieces, and
    come back. The frames differ in a strip under the cue, which the model covers on its own."""
    ctx, st, fmt, n = gctx, 4020, "BGRA", 4
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    rl = [dict(pixels=overlay("translucent", W8, 2700)[:1500], x=0, y=200)]
    frame = random_frame(fmt, W8, H8, 13)
    want = model_blend(fmt, W8, H8, copy_planes(frame), rl)
    frames, wants = [], []
    for k in range(n):
        f = copy_planes(frame)
        f[0][:, 4 * 64 * k:4 * 64 * (k + 1)] ^= np.uint8(17 * (k + 1))
        strip = [f[0][200:1700, 4 * 64 * k:4 * 64 * (k + 1)].copy()]
        strip = model_blend(fmt, 64, 1500, strip, [dict(rl[0], pixels=rl[0]["pixels"][:, 64 * k:64 * (k + 1)], y=0)])
        wk = copy_planes(want)
        wk[0][:, 4 * 64 * k:4 * 64 * (k + 1)] = f[0][:, 4 * 64 * k:4 * 64 * (k + 1)]
        wk[0][200:1700, 4 * 64 * k:4 * 64 * (k + 1)] = strip[0]
        frames.append(f)
        wants.append(wk)
    ctx.overlay_set_rectangles(st, rl)
    if not KNOB:
        assert split(layout_jobs(hooks, fmt, W8, H8, boxes(rl), True))
    hosts = [ctx.acquire(fmt, W8, H8, on_host=True) for _ in range(n)]
    ctx.set_batch(n, 0)
    ctx.set_host_dma(1)
    try:
        for hf, f in zip(hosts, frames):
            hf.host_planes()[0][...] = f[0]
        s0 = ctx.stats()
        tickets = ctx.blend_host_many(tb.TtmlBlend.Batch([st] * n, fmt, W8, H8, [h.c for h in hosts],
                                                         [h.c for h in hosts]))
        ctx.flush()
        ctx.wait(tickets[n - 1])
        d = delta(ctx, s0)
        if not KNOB:
            assert d["host_dma_batches"] >= 1 and d["lazy_launches"] == 0, d
        for k, (hf, wk) in enumerate(zip(hosts, wants)):
            assert_planes_equal([np.array(hf.host_planes()[0])], wk, f"host frame {k}")
    finally:
        ctx.set_host_dma(int(os.environ.get("FLUC_TTMLBLEND_HOST_DMA", "2")))
        ctx.set_batch(32, 200)
        for h in hosts:
            h.release()
    clear_and_check(ctx, [st], base)


# ---------------------------------------------------------------------------------------------
# B. table-kernel fallbacks

B_CASES = [("RGBA", 8192, 3000, 1500), ("Y444", 8192, 3000, 1500), ("RGB", 7680, 0, 4096)]


@pytest.mark.parametrize("fmt,w,x,rw", B_CASES)
def test_ungroupable_frames_take_the_table_kernel(gctx, hooks, fmt, w, x, rw):
    """Four frames out of place in one batch under one cue over rows 1080-3240. The frames are
    one frame with the rows outside the cue changed per frame, so one model serves them all."""
    ctx, st, h, n = gctx, 4030 + B_CASES.index((fmt, w, x, rw)), 4320, 4
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    rl = [dict(pixels=overlay("plain", rw, 2160), x=x, y=1080)]
    frame = random_frame(fmt, w, h, 14)
    want = model_blend(fmt, w, h, copy_planes(frame), rl)
    frames, wants = [], []
    for k in range(n):
        f, wk = copy_planes(frame), copy_planes(want)
        for p, q in zip(f, wk):
            p[:1080] ^= np.uint8(k + 1)
            p[3240:] ^= np.uint8(k + 1)
            q[:1080], q[3240:] = p[:1080], p[3240:]
        frames.append(f)
        wants.append(wk)
    ctx.overlay_set_rectangles(st, rl)
    if not KNOB:
        jobs = layout_jobs(hooks, fmt, w, h, boxes(rl), False)
        assert not any(j.grouped for j in jobs) and any(j.flags & hl.JF_FAST for j in jobs)
    srcs = [ctx.acquire(fmt, w, h) for _ in range(n)]
    dsts = [ctx.acquire(fmt, w, h) for _ in range(n)]
    ctx.set_batch(n, 1_000_000)
    try:
        for s, f in zip(srcs, frames):
            s.upload(f)
        ctx.sync()
        s0 = ctx.stats()
        tickets = ctx.submit_many(tb.TtmlBlend.Batch([st] * n, fmt, w, h, [s.c for s in srcs], [d.c for d in dsts]))
        ctx.flush()
        ctx.wait(tickets[n - 1])
        d = delta(ctx, s0)
        if not KNOB:
            assert d["launches"] > d["group_launches"] + d["multi_launches"], d
        for k, (dst, wk) in enumerate(zip(dsts, wants)):
            assert_planes_equal(dst.download(), wk, f"{fmt} frame {k}")
    finally:
        ctx.set_batch(32, 200)
        for f in srcs + dsts:
            f.release()
    clear_and_check(ctx, [st], base)


# ---------------------------------------------------------------------------------------------
# C. near the limit

C_CASES = [("BGRA", 32764, 1024, 102, 819, ("out", "inplace")),
           ("AYUV", 32764, 1024, 102, 256, ("out", "inplace")),
           ("GRAY8", 32767, 512, 100, 300, ("out", "inplace", "staged")),
           ("I420", 32767, 512, 100, 300, ("out", "inplace", "staged")),
           ("RGBA", 15360, 8640, 2000, 1000, ("out", "inplace"))]


@pytest.mark.parametrize("fmt,w,h,y,rh,modes", C_CASES, ids=[f"{c[0]}-{c[1]}x{c[2]}" for c in C_CASES])
def test_near_the_width_limit(gctx, hooks, fmt, w, h, y, rh, modes):
    """A full-width rectangle: 64-row pieces at 8191 vectors a row (32764 BGRA out of place as group
    bands, in place on the table kernel), a ragged last vector column at 32767 (byte kernel beside
    the group launch), 312-row pieces at 15360 RGBA (table kernel out of place, group in place)."""
    ctx, st = gctx, 4040 + [c[0] for c in C_CASES].index(fmt)
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    rl = [dict(pixels=overlay("plain", w, rh), x=0, y=y)]
    frame = random_frame(fmt, w, h, 15)
    want = model_blend(fmt, w, h, copy_planes(frame), rl)
    ctx.overlay_set_rectangles(st, rl)
    for mode in modes:
        s0 = ctx.stats()
        got = blend(ctx, st, fmt, w, h, frame, mode)
        d = delta(ctx, s0)
        assert_planes_equal(got, want, f"{fmt} {w}x{h} {mode}")
        if KNOB or mode == "staged":
            continue
        jobs = layout_jobs(hooks, fmt, w, h, boxes(rl), mode == "inplace")
        grouped = any(j.grouped for j in jobs)
        table = any(not j.grouped for j in jobs)
        assert (d["group_launches"] + d["multi_launches"] >= 1) == grouped, (mode, d)
        assert (d["launches"] > d["group_launches"] + d["multi_launches"]) == table, (mode, d)
        if w == 32767:
            assert any(j.win_v0 == 2047 and j.win_nv == 1 and not j.flags & hl.JF_FAST for j in jobs)
            assert grouped and table
        else:
            assert split(jobs)
        if (fmt, mode) == ("BGRA", "out"):
            assert grouped and not table
        if (fmt, mode) in (("BGRA", "inplace"), ("RGBA", "out")):
            assert table and not grouped
    clear_and_check(ctx, [st], base)


# ---------------------------------------------------------------------------------------------
# D. offsets past 2^31 and 2^32

D_RECTS = ((0, 0, 256, 64), (16, 16320, 224, 128), (0, 32720, 256, 48))     # top, across 16384, beyond 2^32


def _rows_between(h, spans):
    """Row ranges of [0, h) outside the given (y0, y1) spans."""
    out, y = [], 0
    for y0, y1 in sorted(spans):
        if y0 > y:
            out.append((y, y0))
        y = max(y, y1)
    if y < h:
        out.append((y, h))
    return out


@pytest.mark.parametrize("stride", [2 ** 17 + 256, 2 ** 17 + 259], ids=["aligned", "byte-path"])
@pytest.mark.parametrize("fmt", ["GRAY8", "NV12"])
@pytest.mark.parametrize("mode", ["out", "inplace"])
def test_offsets_past_4_gib(gctx, fmt, stride, mode):
    """256 x 32768 frames whose planes are more than 4 GiB long. Rows under the rectangles are
    downloaded and compared with the model; every other row is compared on the device with the
    source (out of place) or with a copy taken before the blend (in place)."""
    ctx, st, w, h = gctx, 4050, 256, 32768
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    n_planes = 2 if fmt == "NV12" else 1
    assert D_RECTS[2][1] * stride >= 2 ** 32
    g = torch.Generator(device="cuda").manual_seed(16 + stride % 7)
    src = TorchFrame(fmt, w, h, strides=[stride] * n_planes)
    src.buf.random_(0, 256, generator=g)
    dst = src if mode == "inplace" else TorchFrame(fmt, w, h, strides=[stride] * n_planes, fill=0xA5)
    before = src.buf.clone() if mode == "inplace" else src.buf
    rl = [dict(pixels=random_overlay(rw, rh, 300 + k), x=x, y=y) for k, (x, y, rw, rh) in enumerate(D_RECTS)]
    sub = 2 if fmt == "NV12" else 1
    spans = [[(y // (1 if p == 0 else sub), (y + rh) // (1 if p == 0 else sub)) for (_, y, _, rh) in D_RECTS]
             for p in range(n_planes)]
    rows_of = lambda fr, k: [fr.views()[p][spans[p][k][0]:spans[p][k][1]].cpu().numpy() for p in range(n_planes)]
    # the rectangles' rows alone: the model of a rectangle at y = 0 on them (y is even, so the
    # chroma rows of NV12 line up)
    wants = [model_blend(fmt, w, rh, rows_of(src, k), [dict(r, y=0)]) for k, ((_, _, _, rh), r) in
             enumerate(zip(D_RECTS, rl))]
    ctx.overlay_set_rectangles(st, rl)
    note_mem()
    torch.cuda.synchronize()
    ctx.wait(ctx.submit(st, fmt, w, h, src.c, dst.c))
    for k, want in enumerate(wants):
        assert_planes_equal(rows_of(dst, k), want, f"{fmt} stride {stride} {mode} rectangle {k}")
    off = 0
    for p, (s, (rb, rows)) in enumerate(zip(src.strides, src.layout)):
        ref_p = before[off:off + s * rows].view(rows, s)
        for a, b in _rows_between(rows, spans[p]):
            assert torch.equal(dst.planes[p][a:b, :rb], ref_p[a:b, :rb]), (fmt, stride, mode, p, a, b)
        if mode == "inplace":
            assert torch.equal(dst.planes[p][:, rb:], ref_p[:, rb:]), "bytes past the row written"
        off += s * rows
    if mode == "out":
        assert dst.padding_is(0xA5)
    del src, dst, before
    clear_and_check(ctx, [st], base)


def test_32768_square_frame_in_place(gctx):
    """One 32768 x 32768 BGRA frame (stride 2^17 + 256, 4.3 GB) in place under one frame-sized
    straight-alpha rectangle whose pixels are a device tensor (4 GiB; the prepared plane is 4 GiB
    too). 68 sampled rows, among them 0, 16383, 16384 and the last, are compared with the model;
    the bytes past each row are compared on the device with a copy."""
    ctx, st, n = gctx, 4060, 32768
    stride = 2 ** 17 + 256
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    g = torch.Generator(device="cuda").manual_seed(17)
    frame = TorchFrame("BGRA", n, n, strides=[stride])
    frame.buf.random_(0, 256, generator=g)
    pad_before = frame.planes[0][:, 4 * n:].clone()
    rows = sorted({0, 1, 16383, 16384, 32703, 32704, 32705, n - 2, n - 1} |
                  set(np.random.default_rng(18).integers(0, n, 59).tolist()))
    assert len(rows) >= 64
    idx = torch.tensor(rows, device="cuda")
    before = frame.planes[0][idx, :4 * n].cpu().numpy()
    px = torch.empty((n, n, 4), dtype=torch.uint8, device="cuda").random_(0, 256, generator=g)
    ov_rows = px[idx].cpu().numpy()
    r = tb.Rectangle(px.data_ptr(), n, n, 4 * n, 0, 0, 1.0, 0, 0, 0)
    note_mem()
    torch.cuda.synchronize()
    ctx._check(ctx.lib.fluc_ttmlblend_overlay_set_rectangles(ctx.h, st, C.byref(r), 1), "overlay_set_rectangles")
    ctx.sync()
    note_mem()
    del px                          # the library holds its own copy
    torch.cuda.empty_cache()
    ctx.wait(ctx.submit(st, "BGRA", n, n, frame.c, frame.c))
    note_mem()
    got = frame.planes[0][idx, :4 * n].cpu().numpy()
    for i, y in enumerate(rows):
        want = model_blend("BGRA", n, 1, [before[i:i + 1].copy()],
                           [dict(pixels=ov_rows[i:i + 1], x=0, y=0, premultiplied=False)])
        assert_planes_equal([got[i:i + 1]], want, f"row {y}")
    assert torch.equal(frame.planes[0][:, 4 * n:], pad_before), "bytes past the row written"
    del frame, pad_before, idx
    clear_and_check(ctx, [st], base)


# ---------------------------------------------------------------------------------------------
# E. a move at 8K

@pytest.mark.parametrize("place", ["out", "inplace"])
def test_8k_move_shifts_the_piece_boundaries(gctx, hooks, place):
    ctx, fmt, st = gctx, "BGRA", 4070
    ctx.sync()
    base = ctx.stats()["cache_bytes"]
    frame = random_frame(fmt, W8, H8, 19)
    rl = cue_8k(fmt, "plain")
    ctx.overlay_set_rectangles(st, rl)
    blend(ctx, st, fmt, W8, H8, frame, place)
    xs, ys = [3, 2000], [237, rl[1]["y"]]
    moved = [dict(r, x=x, y=y) for r, x, y in zip(rl, xs, ys)]
    ctx.overlay_set_positions(st, xs, ys)
    want = model_blend(fmt, W8, H8, copy_planes(frame), moved)
    if not KNOB:
        jobs = layout_jobs(hooks, fmt, W8, H8, boxes(moved), True)
        assert split(jobs) and any(j.win_y0 == 237 + max_rows(j.win_nv) for j in jobs)
    for pad in (0, 256):
        assert_planes_equal(blend(ctx, st, fmt, W8, H8, frame, place, pad), want, f"moved {place} pad {pad}")
    ctx.overlay_set_rectangles(st + 1, moved)
    for mode, pad in ((place, 256),):
        assert_planes_equal(blend(ctx, st + 1, fmt, W8, H8, frame, mode, pad), want, f"fresh install {mode}")
    clear_and_check(ctx, [st, st + 1], base)
