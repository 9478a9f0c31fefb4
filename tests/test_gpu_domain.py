"""The blend operators over their whole 8-bit domain, through the C ABI, on every kernel path.

Each domain frame is laid out so that every input tuple an operator takes occurs at least once,
and every test first decodes its inputs back from the frame and overlay it hands to the library
and asserts that count (2^24 (alpha, Cs, Cd) triples, 65 536 (a, ga) pairs, ...): a layout bug
cannot shrink a domain unnoticed. The reference is helpers.model_blend (the int64 numpy
restatement of BLENDSPEC sections 2-3), computed once per input; every path's output is
compared with it at tolerance 0, and on a crop the CPU oracle is checked against it too.

D1  OVER at an opaque destination, straight source (blend4_plane8): RGB frames, every
    (asrc, Cs, Cd);
D2  premultiplied source on RGB, ga 255 (the saturating-add branch of blend4_rgb24), Cs > a
    included;
D3  premultiplied source on RGB at ga 1, 127, 254 (the byte loop of blend4_rgb24), set by fades;
D4  asrc = a*ga/255 for every (a, ga): per-frame fades (scale4_alpha; batches of 4, 28 and 64
    frames: the three group parameter blocks) and rectangles installed at that value (folded
    by the prepare kernel);
D5  the packed operators (blend_px_packed*, blend16_packed): every (a, adst, Cd) with every
    Cs, straight / premultiplied source and destination, BGRA (alpha byte 3) and ARGB (byte 0),
    at ga 255 on the full grid and at ga 1, 128, 254 on every (a, adst) pair;
D6  the prepare's un-premultiply and BT.709 matrix (bgra_to_ayuv): every (r, g, b) at alpha 255
    on AYUV, every (a, c) through the un-premultiply, NV12 and GRAY8 luma on a crop.

Every domain frame holds 16-byte vectors whose overlay alpha is all 0, all 255 and mixed (the
middle of each domain is scrambled by an odd multiplier), D5 also destination-alpha vectors all
255 and mixed (with alpha 255 in the first pixel only). Full domains run on the default path;
the kernel paths (TMA-staged one-rectangle bulk, general windows, lazy and opaque-skip variants,
the three group parameter blocks, multi-layout launches, the table kernel with and without
register staging, the byte-granular path) each run a reduced slice that still holds every
(asrc, Cd) pair -- every (a, adst) pair for D5 --, at ga 255 and under a fade, and each asserts
from the context's counters that it ran. Knobs the library reads once per process run in a
child process."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import assert_planes_equal, copy_planes, model_blend, oracle_blend, pkg, wl
from helpers import _matrix_rgb_to_yuv

pytestmark = pytest.mark.gpu

tbm = pkg.ttmlblend
# tools/knob_matrix.sh runs this file with each path knob forced: the counters that prove a path
# ran are only asserted where the environment leaves that path on
GROUPS = os.environ.get("FLUC_TTMLBLEND_GROUPS", "1") != "0"
MULTI = GROUPS and os.environ.get("FLUC_TTMLBLEND_MULTI", "1") != "0"
PACKED_AP = {"BGRA": 3, "ARGB": 0}                  # alpha byte of the destination pixel word


def ga_float(k):
    """The float32 global alpha the library turns into exactly k ((int) (255.0 * value)):
    k / 255 itself can land on k - 1."""
    f = np.float32(k / 255)
    while int(255.0 * float(f)) < k:
        f = np.nextafter(f, np.float32(2))
    assert int(255.0 * float(f)) == k
    return float(f)


def ga_int(f):
    return int(255.0 * float(np.float32(f)))


def scrambled(n):
    """Pixel order: the first and last quarters in order (uniform vectors: all-transparent,
    all-opaque), a power-of-two window in the middle permuted by an odd multiplier (mixed
    vectors)."""
    order = np.arange(n)
    span = 1 << int(np.log2(max(n // 2, 1)))
    lo = (n - span) // 2
    order[lo:lo + span] = lo + (np.arange(span, dtype=np.int64) * 0x9E3779B1) % span
    assert np.array_equal(np.sort(order), np.arange(n))
    return order


def lay_out(cols, w):
    """Per-pixel columns (N, ...) -> (rows, w, ...) in scrambled order, padded with zeros."""
    n = cols.shape[0]
    rows = -(-n // w)
    out = np.zeros((rows * w,) + cols.shape[1:], cols.dtype)
    out[:n] = cols[scrambled(n)]
    return out.reshape((rows, w) + cols.shape[1:])


def model_banded(fmt, w, h, planes, rects, dp=False, band=512):
    """model_blend of one frame-sized rectangle at the origin, in row bands (bounded memory)."""
    planes = copy_planes(planes)
    for y0 in range(0, h, band):
        y1 = min(h, y0 + band)
        sub = [p[y0:y1] for p in planes]
        model_blend(fmt, w, y1 - y0, sub, [dict(r, pixels=r["pixels"][y0:y1]) for r in rects], dp)
    return planes


def check_oracle_crop(fmt, w, frame, rects, want, dp=False, rows=256):
    """The CPU oracle agrees with the reference on the first rows."""
    crop = [p[:rows].copy() for p in frame]             # the oracle blends in place
    got = oracle_blend(fmt, w, rows, crop, [dict(r, pixels=np.ascontiguousarray(r["pixels"][:rows]))
                                            for r in rects], dp)
    assert_planes_equal(got, [p[:rows] for p in want], f"oracle on a crop of {fmt}")


def run(ctx, stream, fmt, w, h, frame, mode="out", dp=False):
    flags = tbm.FLAG_PREMULTIPLIED_ALPHA if dp else 0
    src = ctx.acquire(fmt, w, h)
    try:
        src.upload(frame)
        if mode == "inplace":
            ctx.wait(ctx.submit(stream, fmt, w, h, src.c, src.c, flags))
            return src.download()
        dst = ctx.acquire(fmt, w, h)
        try:
            ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dst.c, flags))
            return dst.download()
        finally:
            dst.release()
    finally:
        src.release()


def delta(ctx, before):
    now = ctx.stats()
    return {k: now[k] - before[k] for k in now}


# ---------------------------------------------------------------------------
# domain frames

class Dom:
    """A domain frame: format, size, frame planes, overlay image (one frame-sized rectangle)."""

    def __init__(self, fmt, frame, img, sp):
        self.fmt, self.frame, self.img, self.sp = fmt, frame, img, sp
        self.h, self.w = img.shape[:2]

    def rects(self, ga=1.0):
        return [dict(pixels=self.img, x=0, y=0, global_alpha=ga, premultiplied=self.sp)]

    def want(self, ga=1.0, dp=False):
        return model_banded(self.fmt, self.w, self.h, self.frame, self.rects(ga), dp)


def rgb_dom(fmt, w, sp, full=True):
    """D1-D3 on a 24-bit RGB frame: the three bytes of a pixel share its alpha and carry their
    own (Cs, Cd). full: every (a, Cs, Cd); else every (a, Cd) with Cs a function of both."""
    per = 21846 if full else 86                   # pixels per alpha: 3 * per >= 65536 / 256 slots
    q = np.arange(256 * per)
    a = q // per
    m = (3 * (q % per))[:, None] + np.arange(3)
    if full:
        m %= 65536
        cs, cd = m >> 8, m & 255
    else:
        cd = m % 256
        cs = (cd * 167 + a[:, None] * 73 + 11) & 255
    px = np.zeros((q.size, 4), np.uint8)
    px[:, 2], px[:, 1], px[:, 0] = cs[:, 0], cs[:, 1], cs[:, 2]     # R, G, B of the BGRA word
    px[:, 3] = a
    dst = cd.astype(np.uint8)
    order = (0, 1, 2) if fmt == "RGB" else (2, 1, 0)
    dst = dst[:, order]
    img = lay_out(px, w)
    frame = [lay_out(dst, w).reshape(img.shape[0], 3 * w)]
    return Dom(fmt, frame, img, sp)


def rgb_coverage(d, full=True):
    """Decoded from what the library gets: (a, Cs, Cd) per destination byte."""
    a = d.img[..., 3].astype(np.int64)
    rgb = d.img[..., [2, 1, 0]].astype(np.int64)
    if d.fmt == "BGR":
        rgb = rgb[..., ::-1]
    cd = d.frame[0].reshape(d.h, d.w, 3).astype(np.int64)
    key = (a[..., None] << 16) | (rgb << 8) | cd if full else (a[..., None] << 8) | cd
    return distinct(key)


def distinct(key):
    return int(np.count_nonzero(np.bincount(key.ravel())))


def packed_dom(fmt, w, sp, full=True):
    """D5: every (a, adst, Cd) (full) or every (a, adst) with Cd a function (slice); the three
    colour channels take different bijections of Cd for Cs and Cd, so that every Cs meets every
    (a, adst). The first half keeps its order: uniform vectors of overlay and destination alpha;
    the middle is scrambled; rows at the end have adst 255 in the first pixel of a vector only."""
    n = 1 << 24 if full else 1 << 16
    t = np.arange(n, dtype=np.int64)
    if full:
        a, adst, cd = t >> 16, (t >> 8) & 255, t & 255
    else:
        a, adst = t >> 8, t & 255
        cd = (a * 29 + adst * 101 + 7) & 255
    cs = np.stack([(cd * 7 + 3) & 255, (cd * 13 + 5) & 255, (cd * 11 + 1) & 255], 1)
    cdc = np.stack([cd, (cd + 85) & 255, (cd * 3 + 170) & 255], 1)
    ap = PACKED_AP[fmt]
    cpos = [k for k in range(4) if k != ap]
    # the overlay: BGRA words (straight or premultiplied colours are just bytes here)
    px = np.zeros((n, 4), np.uint8)
    px[:, 0], px[:, 1], px[:, 2], px[:, 3] = cs[:, 2], cs[:, 1], cs[:, 0], a   # B G R A
    # the destination word: c1 c2 c3 = R G B in the format's byte order
    order = {"BGRA": (2, 1, 0), "ARGB": (0, 1, 2)}[fmt]          # channel of each colour byte
    dw = np.zeros((n, 4), np.uint8)
    dw[:, ap] = adst
    for pos, ch in zip(cpos, order):
        dw[:, pos] = cdc[:, ch]
    img = lay_out(px, w)
    dst = lay_out(dw, w)
    # extra rows: destination-alpha vectors alternately all 255 and mixed with 255 in the first
    # pixel only
    tail = 16
    extra = dst[:tail].copy().reshape(-1, 4)
    k = np.arange(extra.shape[0])
    extra[:, ap] = np.where((k % 8 < 4) | (k % 4 == 0), 255, (k * 37) % 255)
    img = np.concatenate([img, img[-tail:]])
    dst = np.concatenate([dst, extra.reshape(tail, w, 4)])
    return Dom(fmt, [dst.reshape(img.shape[0], 4 * w)], img, sp)


def packed_coverage(d, full=True):
    ap = PACKED_AP[d.fmt]
    a = d.img[..., 3].astype(np.int64)
    fw = d.frame[0].reshape(d.h, d.w, 4).astype(np.int64)
    adst = fw[..., ap]
    cd = fw[..., 2 if d.fmt == "BGRA" else 1]                      # the R byte
    key = (a << 16) | (adst << 8) | cd if full else (a << 8) | adst
    return distinct(key)


def assert_vectors(d, packed=False):
    """The frame holds 16-byte overlay vectors with alpha all 0, all 255 and mixed (and, packed,
    destination-alpha vectors all 255 and mixed)."""
    if packed:
        oa = d.img[..., 3][:, :d.w // 4 * 4].reshape(-1, 4)
        fa = d.frame[0].reshape(d.h, d.w, 4)[..., PACKED_AP[d.fmt]][:, :d.w // 4 * 4].reshape(-1, 4)
        assert (fa == 255).all(1).any() and ((fa == 255).any(1) & ~(fa == 255).all(1)).any()
        assert ((fa[:, 0] == 255) & (fa[:, 1:] != 255).any(1)).any()
    else:
        rb = 3 * d.w
        oa = np.repeat(d.img[..., 3], 3, axis=1)[:, :rb // 16 * 16].reshape(-1, 16)
    assert (oa == 0).all(1).any() and (oa == 255).all(1).any()
    assert ((oa != 0).any(1) & (oa != oa[:, :1]).any(1)).any()


# ---------------------------------------------------------------------------
# D1 - D3: RGB

@pytest.mark.parametrize("fmt,w", [("RGB", 2048), ("BGR", 2045)])      # 2045 * 3: ragged rows
@pytest.mark.parametrize("sp", [False, True])
def test_rgb_over_whole_domain(ctx, fmt, w, sp):
    """D1 (straight) / D2 (premultiplied, Cs > a included): every (asrc, Cs, Cd) at ga 255, in
    and out of place."""
    d = rgb_dom(fmt, w, sp)
    assert rgb_coverage(d) == 1 << 24
    assert_vectors(d)
    want = d.want()
    check_oracle_crop(fmt, d.w, d.frame, d.rects(), want)
    ctx.overlay_set_rectangles(300, d.rects())
    for mode in ("out", "inplace"):
        assert_planes_equal(run(ctx, 300, fmt, d.w, d.h, d.frame, mode), want, f"{fmt} sp={sp} {mode}")


def test_rgb_premultiplied_faded_whole_domain(ctx):
    """D3: the byte loop of blend4_rgb24, MIN (255, (Cs*ga + Cd*(255-asrc)) / 255), at ga 1, 127
    and 254 set by fades of a rectangle installed at 1."""
    d = rgb_dom("RGB", 2048, True)
    assert rgb_coverage(d) == 1 << 24
    ctx.overlay_set_rectangles(301, d.rects())
    run(ctx, 301, "RGB", d.w, d.h, d.frame)                       # prepared at 1
    for k in (1, 127, 254):
        f = ga_float(k)
        ctx.overlay_set_global_alpha(301, f)
        want = d.want(f)
        if k == 127:
            check_oracle_crop("RGB", d.w, d.frame, d.rects(f), want)
        st = ctx.stats()
        assert_planes_equal(run(ctx, 301, "RGB", d.w, d.h, d.frame), want, f"ga={k}")
        assert delta(ctx, st)["prepare_launches"] == 0


# ---------------------------------------------------------------------------
# D4: asrc = a * ga / 255

D4_W = 256


def d4_rows():
    """4 rows of a in 0..255: ascending (mixed vectors), 0, 255, descending; Cs 255, straight."""
    a = np.stack([np.arange(256), np.zeros(256, int), np.full(256, 255), 255 - np.arange(256)])
    img = np.full((4, D4_W, 4), 255, np.uint8)
    img[..., 3] = a
    return img


def test_global_alpha_scaling_as_fades(ctx):
    """Every (a, ga) as per-frame fades of one rectangle: over Cd = 0 with Cs = 255 the output
    byte is asrc itself. Batches of 4, 28 and 64 frames in one launch each (the three group
    parameter blocks), ga 0 on its own (no band: the copy)."""
    img = np.concatenate([d4_rows()] * 4)
    h = img.shape[0]
    rl = [dict(pixels=img, x=0, y=0, premultiplied=False)]
    frame = [np.zeros((h, 3 * D4_W), np.uint8)]
    ctx.overlay_set_rectangles(310, rl)
    run(ctx, 310, "RGB", D4_W, h, frame)
    src = ctx.acquire("RGB", D4_W, h)
    src.upload(frame)
    seen = set()
    values = list(range(1, 256))
    batches = [4, 28, 64, 64, 64, 31]
    assert sum(batches) == len(values)
    ctx.set_batch(64, 1_000_000)
    try:
        for n in batches:
            ks, values = values[:n], values[n:]
            dsts = [ctx.acquire("RGB", D4_W, h) for _ in ks]
            st = ctx.stats()
            tickets = []
            for k, dst in zip(ks, dsts):
                ctx.overlay_set_global_alpha(310, ga_float(k))
                tickets.append(ctx.submit(310, "RGB", D4_W, h, src.c, dst.c))
            ctx.flush()
            for t in tickets:
                ctx.wait(t)
            dl = delta(ctx, st)
            assert dl["launches"] == 1 and dl["group_launches"] == (1 if GROUPS else 0), (n, dl)
            assert dl["prepare_launches"] == 0
            for k, dst in zip(ks, dsts):
                got = dst.download()[0].reshape(h, D4_W, 3)
                asrc = img[..., 3].astype(np.int64) * k // 255
                assert np.array_equal(got, np.repeat(asrc[..., None], 3, 2)), k
                seen.update(zip(img[..., 3].ravel().tolist(), [k] * img[..., 3].size))
                dst.release()
    finally:
        ctx.set_batch(32, 200)
    ctx.overlay_set_global_alpha(310, 0.0)
    assert_planes_equal(run(ctx, 310, "RGB", D4_W, h, frame), frame, "ga 0")
    seen.update((a, 0) for a in range(256))
    src.release()
    assert len(seen) == 1 << 16
    want = model_blend("RGB", D4_W, h, copy_planes(frame), faded_rects(rl, ga_float(200)))
    ctx.overlay_set_global_alpha(310, ga_float(200))
    assert_planes_equal(run(ctx, 310, "RGB", D4_W, h, frame), want, "model at 200")


def faded_rects(rl, ga):
    return [dict(r, global_alpha=ga) for r in rl]


def test_global_alpha_scaling_folded(ctx):
    """Every (a, ga) folded by the prepare kernel: 64 rectangles per install, each at its own
    value, four installs."""
    h = 4 * 64
    frame = [np.zeros((h, 3 * D4_W), np.uint8)]
    seen = set()
    for part in range(4):
        ks = list(range(64 * part, 64 * part + 64))
        rl = [dict(pixels=d4_rows(), x=0, y=4 * j, global_alpha=ga_float(k) if k else 0.0, premultiplied=False)
              for j, k in enumerate(ks)]
        assert [ga_int(r["global_alpha"]) for r in rl] == ks
        ctx.overlay_set_rectangles(311, rl)
        got = run(ctx, 311, "RGB", D4_W, h, frame)[0].reshape(h, D4_W, 3)
        for j, k in enumerate(ks):
            a = d4_rows()[..., 3].astype(np.int64)
            assert np.array_equal(got[4 * j:4 * j + 4], np.repeat((a * k // 255)[..., None], 3, 2)), k
            seen.update((int(x), k) for x in np.unique(a))
        assert_planes_equal([got.reshape(h, -1)], model_blend("RGB", D4_W, h, copy_planes(frame), rl), "model")
    assert len(seen) == 1 << 16


# ---------------------------------------------------------------------------
# D5: packed

@functools.lru_cache(maxsize=1)
def packed_full(fmt):
    return packed_dom(fmt, 4096, False)


@pytest.mark.parametrize("dp", [False, True])
@pytest.mark.parametrize("sp", [False, True])
@pytest.mark.parametrize("fmt", list(PACKED_AP))
def test_packed_whole_domain(ctx, fmt, sp, dp):
    """D5 at ga 255: every (a, adst, Cd), every Cs against every (a, adst)."""
    d = packed_full(fmt)
    d = Dom(fmt, d.frame, d.img, sp)
    assert packed_coverage(d) == 1 << 24
    assert_vectors(d, packed=True)
    want = d.want(dp=dp)
    if not sp:
        check_oracle_crop(fmt, d.w, d.frame, d.rects(), want, dp, rows=64)
    ctx.overlay_set_rectangles(320, d.rects())
    assert_planes_equal(run(ctx, 320, fmt, d.w, d.h, d.frame, dp=dp), want, f"{fmt} sp={sp} dp={dp}")


@pytest.mark.parametrize("fmt", list(PACKED_AP))
def test_packed_faded_every_alpha_pair(ctx, fmt):
    """D5 at ga 1, 128, 254: every (a, adst) with 16 values of Cd each, sp x dp."""
    for sp in (False, True):
        d = packed_dom(fmt, 1024, sp, full=False)
        # 16 Cd values per (a, adst): the slice's Cd, stepped through 16 offsets row band by band
        frames = []
        for off in range(16):
            f = d.frame[0].reshape(d.h, d.w, 4).copy()
            for pos in range(4):
                if pos != PACKED_AP[fmt]:
                    f[..., pos] = (f[..., pos].astype(np.int64) + 16 * off) & 255
            frames.append([f.reshape(d.h, 4 * d.w)])
        assert packed_coverage(d, full=False) == 1 << 16
        cds = set()
        for f in frames:
            cds.update(np.unique(f[0].reshape(d.h, d.w, 4)[..., 2 if fmt == "BGRA" else 1]).tolist())
        assert len(cds) == 256
        ctx.overlay_set_rectangles(321, d.rects())
        run(ctx, 321, fmt, d.w, d.h, frames[0])
        for k in (1, 128, 254):
            ctx.overlay_set_global_alpha(321, ga_float(k))
            for dp in (False, True):
                for i, f in enumerate(frames):
                    want = model_blend(fmt, d.w, d.h, copy_planes(f), d.rects(ga_float(k)), dp)
                    assert_planes_equal(run(ctx, 321, fmt, d.w, d.h, f, dp=dp), want, f"ga={k} sp={sp} dp={dp} {i}")


# ---------------------------------------------------------------------------
# D6: the prepare's matrix and un-premultiply

def test_matrix_every_rgb(ctx):
    """Every (r, g, b) at alpha 255 onto AYUV (ga 255, opaque frame): the output pixel is the
    BT.709 matrix output itself; straight and premultiplied (at 255 the un-premultiply is the
    identity). A transparent and a mixed band below give the other vector kinds."""
    t = np.arange(1 << 24, dtype=np.int64)
    r, g, b = t >> 16, (t >> 8) & 255, t & 255
    w, hd = 4096, 4096
    img = np.zeros((hd + 16, w, 4), np.uint8)
    img[:hd, :, 0] = b.reshape(hd, w)
    img[:hd, :, 1] = g.reshape(hd, w)
    img[:hd, :, 2] = r.reshape(hd, w)
    img[:hd, :, 3] = 255
    img[hd + 8:, :, 3] = np.arange(w) % 256
    img[hd + 8:, :, :3] = (np.arange(w) * 7 % 256)[:, None]
    key = (img[:hd, :, 2].astype(np.int64) << 16) | (img[:hd, :, 1].astype(np.int64) << 8) | img[:hd, :, 0]
    assert distinct(key) == 1 << 24
    h = hd + 16
    frame = [np.full((h, 4 * w), 77, np.uint8)]
    frame[0][:, 0::4] = 255
    y, u, v = _matrix_rgb_to_yuv(r, g, b)
    for sp in (False, True):
        rl = [dict(pixels=img, x=0, y=0, premultiplied=sp)]
        want = frame[0].copy()
        body = want[:hd].reshape(hd, w, 4)
        body[..., 0], body[..., 1], body[..., 2], body[..., 3] = 255, y.reshape(hd, w), u.reshape(hd, w), \
            v.reshape(hd, w)
        tail = [frame[0][hd:].copy()]                         # model_blend blends in place
        model_blend("AYUV", w, 16, tail, [dict(pixels=img[hd:], premultiplied=sp)])
        want[hd:] = tail[0]
        check_oracle_crop("AYUV", w, frame, rl, [want], rows=64)
        ctx.overlay_set_rectangles(330, rl)
        assert_planes_equal(run(ctx, 330, "AYUV", w, h, frame), [want], f"sp={sp}")


@pytest.mark.parametrize("fmt", ["AYUV", "NV12", "GRAY8"])
def test_unpremultiply_every_alpha_colour(ctx, fmt):
    """Every (a, c) through (c*255 + a/2) / a: c on R, (c + 85) on G, (c + 170) on B, so each
    channel sees every pair; the result is blended over a frame that keeps it visible."""
    a, c = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    img = np.zeros((256, 256, 4), np.uint8)
    img[..., 3] = a
    img[..., 2], img[..., 1], img[..., 0] = c, (c + 85) % 256, (c + 170) % 256
    assert np.unique((img[..., 3].astype(np.int64) << 8) | img[..., 2]).size == 1 << 16
    w, h = 256, 256
    planes = [np.zeros((rows, rb), np.uint8) for rows, rb in wl.plane_shapes(fmt, w, h)]
    for p in planes:
        p[...] = (np.arange(p.shape[1]) * 5 % 256)[None, :]
    if fmt == "AYUV":
        planes[0][:, 0::4] = 255
    rl = [dict(pixels=img, x=0, y=0)]
    want = model_blend(fmt, w, h, copy_planes(planes), rl)
    assert_planes_equal(oracle_blend(fmt, w, h, copy_planes(planes), rl), want, "oracle")
    ctx.overlay_set_rectangles(331, rl)
    for mode in ("out", "inplace"):
        assert_planes_equal(run(ctx, 331, fmt, w, h, planes, mode), want, f"{fmt} {mode}")


# ---------------------------------------------------------------------------
# kernel paths on reduced slices

SLICES = {"RGB": lambda: rgb_dom("RGB", 200, True, full=False),        # 600-byte rows: ragged
          "RGB_straight": lambda: rgb_dom("RGB", 256, False, full=False),
          "BGRA": lambda: packed_dom("BGRA", 250, False, full=False)}   # 1000-byte rows: ragged
FADE = ga_float(128)


def slice_checked(name):
    d = SLICES[name]()
    if d.fmt == "BGRA":
        assert packed_coverage(d, full=False) == 1 << 16
        assert_vectors(d, packed=True)
    else:
        assert rgb_coverage(d, full=False) == 1 << 16
        assert_vectors(d)
    return d


def general_rects(d, ga=1.0):
    """Two overlapping partial-width rectangles."""
    a, b = d.w * 2 // 3, d.w // 3
    return [dict(pixels=np.ascontiguousarray(d.img[:, :a]), x=0, y=0, global_alpha=ga, premultiplied=d.sp),
            dict(pixels=np.ascontiguousarray(d.img[::-1, b:]), x=b, y=0, global_alpha=ga, premultiplied=d.sp)]


def want_of(d, rl, dp=False):
    return model_blend(d.fmt, d.w, d.h, copy_planes(d.frame), rl, dp)


def install(ctx, stream, d, rl, fade):
    """rl installed at 1 and blended once (prepared), then faded to `fade` when given."""
    ctx.overlay_set_rectangles(stream, rl)
    run(ctx, stream, d.fmt, d.w, d.h, d.frame)
    if fade is not None:
        ctx.overlay_set_global_alpha(stream, fade)
        rl = faded_rects(rl, fade)
    return rl


def batch_run(ctx, streams, d, n_frames=None):
    """Frames of `streams` (one each, or n_frames of streams[0]) submitted together, one flush."""
    streams = streams if n_frames is None else [streams[0]] * n_frames
    src = ctx.acquire(d.fmt, d.w, d.h)
    src.upload(d.frame)
    dsts = [ctx.acquire(d.fmt, d.w, d.h) for _ in streams]
    ctx.set_batch(64, 1_000_000)
    try:
        st = ctx.stats()
        tickets = [ctx.submit(s, d.fmt, d.w, d.h, src.c, dst.c) for s, dst in zip(streams, dsts)]
        ctx.flush()
        for t in tickets:
            ctx.wait(t)
        dl = delta(ctx, st)
        outs = [dst.download() for dst in dsts]
    finally:
        ctx.set_batch(32, 200)
        for f in [src] + dsts:
            f.release()
    return outs, dl


def check_group_paths(ctx, name, fade, base=400, expect=None):
    """One-rectangle bulk and general windows, out of place and in place, and the three group
    parameter blocks (1-4, 5-32, more than 32 frames in one launch). `expect`: counters that must
    move (the knob under test)."""
    d = slice_checked(name)
    one = install(ctx, base, d, d.rects(), fade)
    gen = install(ctx, base + 1, d, general_rects(d), fade)
    moved = {}
    for stream, rl, what in ((base, one, "bulk"), (base + 1, gen, "general")):
        want = want_of(d, rl)
        if fade is None and what == "bulk":
            assert_planes_equal(oracle_blend(d.fmt, d.w, d.h, copy_planes(d.frame), rl), want, "oracle")
        for mode in ("out", "inplace"):
            st = ctx.stats()
            assert_planes_equal(run(ctx, stream, d.fmt, d.w, d.h, d.frame, mode), want, f"{name} {what} {mode}")
            dl = delta(ctx, st)
            assert dl["group_launches"] >= 1 or not GROUPS, (what, mode, dl)
            for k in expect or ():
                moved[k] = moved.get(k, 0) + dl[k]
        for n in (3, 20, 40):
            outs, dl = batch_run(ctx, [stream], d, n)
            assert dl["group_launches"] == (1 if GROUPS else 0), (what, n, dl)   # ragged rows: + a table launch
            for i in (0, n - 1):
                assert_planes_equal(outs[i], want, f"{name} {what} {n} frames, frame {i}")
    for k in expect or ():
        assert moved[k] > 0 or not GROUPS, (k, moved)


@pytest.mark.parametrize("fade", [None, FADE], ids=["ga255", "faded"])
@pytest.mark.parametrize("name", list(SLICES))
def test_group_paths(ctx, name, fade):
    check_group_paths(ctx, name, fade)


@pytest.mark.parametrize("fade", [None, FADE], ids=["ga255", "faded"])
@pytest.mark.parametrize("name", list(SLICES))
def test_multi_layout_launch(ctx, name, fade):
    """Frames of streams with different band lists in one launch."""
    d = slice_checked(name)
    one = install(ctx, 420, d, d.rects(), fade)
    gen = install(ctx, 421, d, general_rects(d), fade)
    outs, dl = batch_run(ctx, [420, 421, 420, 421], d)
    if MULTI:
        assert dl["multi_launches"] == 1 and dl["group_launches"] == 0, dl
    for out, rl in zip(outs, [one, gen, one, gen]):
        assert_planes_equal(out, want_of(d, rl), f"{name} multi")


def test_mixed_fade_kinds_in_one_launch(ctx):
    """One launch holding frames of a faded stream, an unfaded one and one installed at 0.4
    (folded): under the GA variant the unfaded refs are scaled by 255, the identity."""
    d = slice_checked("RGB_straight")
    faded = install(ctx, 430, d, d.rects(), 0.5)
    plain = install(ctx, 431, d, d.rects(), None)
    folded = install(ctx, 432, d, d.rects(0.4), None)
    outs, dl = batch_run(ctx, [430, 431, 432], d)
    assert dl["launches"] == 1 and dl["group_launches"] + dl["multi_launches"] == (1 if GROUPS else 0), dl
    for out, rl in zip(outs, [faded, plain, folded]):
        assert_planes_equal(out, want_of(d, rl), f"ga {rl[0]['global_alpha']}")


@pytest.mark.parametrize("fade", [None, FADE], ids=["ga255", "faded"])
@pytest.mark.parametrize("name", list(SLICES))
def test_table_kernel(monkeypatch, lib, name, fade):
    """FLUC_TTMLBLEND_GROUPS=0: the table kernel (register-staged one-rectangle and general
    windows, byte-granular jobs for the ragged rows)."""
    monkeypatch.setenv("FLUC_TTMLBLEND_GROUPS", "0")
    c = pkg.TtmlBlend(0)
    try:
        d = slice_checked(name)
        for stream, rl in ((440, d.rects()), (441, general_rects(d))):
            rl = install(c, stream, d, rl, fade)
            for mode in ("out", "inplace"):
                st = c.stats()
                assert_planes_equal(run(c, stream, d.fmt, d.w, d.h, d.frame, mode), want_of(d, rl), f"{name} {mode}")
                dl = delta(c, st)
                assert dl["launches"] >= 1 and dl["group_launches"] == 0 and dl["multi_launches"] == 0, dl
    finally:
        c.close()


def run_unaligned(ctx, stream, d):
    """The frame at a 4-byte aligned base with a stride that is a multiple of 4, not of 16."""
    (rows, rb), = wl.plane_shapes(d.fmt, d.w, d.h)
    stride = rb + 4 - (rb % 4) + 4
    big, out = ctx.acquire(d.fmt, d.w + 64, d.h), ctx.acquire(d.fmt, d.w + 64, d.h)
    try:
        src_f, dst_f = tbm.Frame(), tbm.Frame()
        for f, pool in ((src_f, big), (dst_f, out)):
            f.plane[0] = pool.c.plane[0] + 4
            f.stride[0] = stride
        buf = np.zeros((rows, stride), np.uint8)
        buf[:, :rb] = d.frame[0]
        ctx._check(ctx.lib.fluc_ttmlblend_frame_upload(ctx.h, tbm.FORMATS[d.fmt], d.w, d.h,
                                                       tbm._frame_from_arrays([buf[:, :rb]]), src_f), "up")
        ctx.wait(ctx.submit(stream, d.fmt, d.w, d.h, src_f, dst_f))
        got = [np.zeros((rows, rb), np.uint8)]
        ctx._check(ctx.lib.fluc_ttmlblend_frame_download(ctx.h, tbm.FORMATS[d.fmt], d.w, d.h, dst_f,
                                                         tbm._frame_from_arrays(got)), "down")
        return got
    finally:
        big.release()
        out.release()


@pytest.mark.parametrize("fade", [None, FADE], ids=["ga255", "faded"])
@pytest.mark.parametrize("name", list(SLICES))
def test_byte_path(ctx, name, fade):
    """Unaligned base and stride: every window runs byte-granular."""
    d = slice_checked(name)
    for stream, rl in ((450, d.rects()), (451, general_rects(d))):
        rl = install(ctx, stream, d, rl, fade)
        assert_planes_equal(run_unaligned(ctx, stream, d), want_of(d, rl), f"{name} unaligned")


KNOB_CHECK = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import test_gpu_domain as t
c = t.pkg.TtmlBlend(0)
try:
    expect = sys.argv[3].split(",") if sys.argv[3] else None
    for name in t.SLICES:
        for fade in (None, t.FADE):
            t.check_group_paths(c, name, fade, expect=expect)
finally:
    c.close()
print("ok")
"""

KNOBS = [({"FLUC_TTMLBLEND_LAZY": "1"}, "lazy_launches"),
         ({"FLUC_TTMLBLEND_OPAQUE_SKIP": "1"}, "opaque_skip_launches"),
         ({"FLUC_TTMLBLEND_BULK": "0"}, ""),
         ({"FLUC_TTMLBLEND_COMPACT_PARAMS": "0"}, ""),
         ({"FLUC_TTMLBLEND_LANES": "7"}, "")]


@pytest.mark.parametrize("knobs,expect", KNOBS, ids=[next(iter(k)) + "=" + next(iter(k.values())) for k, _ in KNOBS])
def test_group_paths_with_knobs(monkeypatch, knobs, expect):
    """Knobs the library reads once per process, in a child: lazy in place (LAZY 1), opaque skip
    out of place (LAZY 2), register staging instead of the TMA, full-size parameter blocks only,
    interleaved chunk order."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    here = os.path.dirname(os.path.abspath(__file__))
    out = subprocess.run([sys.executable, "-c", KNOB_CHECK, here, os.path.dirname(here), expect],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout + out.stderr
