"""The per-cue kernels against exact models, over their domains and at their edges.

The kernels that build a cue's overlay run once per cue, but whatever they get wrong is blended
into every frame the cue is shown on. Each test here compares one of them, through the C ABI, at
tolerance 0 with an independent model: helpers.model_scale / model_scale_rows, helpers.model_blend
(chroma_average=True), and the restatements below of pixman's MUL_UN8 / OVER / IN, Cairo's colour
conversion and the Gaussian convolution; the C oracle too where it is fast enough. Every domain
test first decodes its input tuples from the pixels it hands over and asserts how many it covers.

Readback: an overlay blended onto an all-zero BGRA frame with FLAG_PREMULTIPLIED_ALPHA comes back
as itself wherever its alpha is above 0 (OVER11 with adst = 0, ga = 255) and as 0 elsewhere;
test_readback_is_the_overlay proves that once on an unscaled control rectangle.

S  ttmlblend_scale_kernel + scale_row_plan: every (a, b, f) of scale_mix_h on each byte lane,
   every (ca, cb, w) of the vertical merge, every source width 2..40 x render width 1..80,
   clipped origins, 1x1, sides of 32768, and the refusal of 32769;
R  ttmlblend_region_kernel: every (s_c, s_a, d_c) of OVER, every (g_c, m8) of the opacity group
   at both ends of every m8 step, every (c, a) of cairo_solid_pixel, layers on regions hanging
   over each frame edge;
B  ttmlblend_blur_kernel: every radius 0..64 on small odd shapes and padded strides, both sides
   of the 48 KB shared-memory boundary, every (v, tap) of impulse images, dst == src;
W  ttmlblend_rowspan_kernel: a visible pixel at every column of widths 1..300, 4096 and 32768
   survives the crop; the lazy / opaque-skip decisions flip exactly at 0.3;
C  ttmlblend_prepare_chroma_avg_kernel: every origin parity, odd and even sizes, clipped edges,
   spans across a 256-thread block, I420 / YV12 / NV12 / NV21;
X  a fade (overlay_set_global_alpha) of a scaled rectangle installed below 1.0 and of a
   region-form overlay."""
import math
import os

import numpy as np
import pytest

from helpers import (assert_planes_equal, copy_planes, model_blend, model_scale, model_scale_rows, oracle_blend, pkg,
                     random_frame, random_overlay)
from oracle import oracle

pytestmark = pytest.mark.gpu

tbm = pkg.ttmlblend
LAZY_KNOBS = ("FLUC_TTMLBLEND_LAZY", "FLUC_TTMLBLEND_OPAQUE_SKIP", "FLUC_TTMLBLEND_GROUPS", "FLUC_TTMLBLEND_MULTI")


def distinct(key):
    return int(np.count_nonzero(np.bincount(np.asarray(key, dtype=np.int64).ravel())))


def run_bgra(ctx, stream, w, h, frame=None, inplace=False):
    """One BGRA frame (all zero by default) blended with FLAG_PREMULTIPLIED_ALPHA; h x w x 4 back."""
    if frame is None:
        frame = np.zeros((h, w, 4), np.uint8)
    src = ctx.acquire("BGRA", w, h)
    try:
        src.upload([frame.reshape(h, 4 * w)])
        if inplace:
            ctx.wait(ctx.submit(stream, "BGRA", w, h, src.c, src.c, tbm.FLAG_PREMULTIPLIED_ALPHA))
            return src.download()[0].reshape(h, w, 4)
        dst = ctx.acquire("BGRA", w, h)
        try:
            ctx.wait(ctx.submit(stream, "BGRA", w, h, src.c, dst.c, tbm.FLAG_PREMULTIPLIED_ALPHA))
            return dst.download()[0].reshape(h, w, 4)
        finally:
            dst.release()
    finally:
        src.release()


def visible(img):
    """What the readback shows of an overlay image: itself where alpha > 0, else 0."""
    return np.where(img[..., 3:4] > 0, img, 0).astype(np.uint8)


def run_fmt(ctx, stream, fmt, w, h, planes):
    """One frame of any format blended out of place with the stream's overlay."""
    src, dst = ctx.acquire(fmt, w, h), ctx.acquire(fmt, w, h)
    try:
        src.upload(planes)
        ctx.wait(ctx.submit(stream, fmt, w, h, src.c, dst.c))
        return dst.download()
    finally:
        src.release()
        dst.release()


def readback_rects(ctx, stream, w, h, rects):
    ctx.overlay_set_rectangles(stream, rects)
    return run_bgra(ctx, stream, w, h)


def model_readback(w, h, rects):
    """helpers.model_blend of the rectangles onto the zero frame, premultiplied destination."""
    return model_blend("BGRA", w, h, [np.zeros((h, 4 * w), np.uint8)], rects, dest_premul=True)[0].reshape(h, w, 4)


def test_readback_is_the_overlay(ctx):
    """The identity the other tests rely on: every (a, c), premultiplied or not (c > a
    included), unscaled, comes back as itself where a > 0 and as 0 where a == 0."""
    a, c = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    img = np.zeros((256, 256, 4), np.uint8)
    img[..., 3] = a
    img[..., 0], img[..., 1], img[..., 2] = c, 255 - c, (c * 7 + a) & 255
    assert distinct((img[..., 3].astype(np.int64) << 8) | img[..., 0]) == 1 << 16
    rl = [dict(pixels=img, x=0, y=0)]
    got = readback_rects(ctx, 500, 256, 256, rl)
    assert np.array_equal(got, visible(img))
    assert np.array_equal(got, model_readback(256, 256, rl))


# ---------------------------------------------------------------------------
# S: the scaler

def x_inc_of(sw, dw):
    return 0 if dw == 1 else ((sw - 1) << 16) // (dw - 1) - 1


def h_mix(a, b, f):
    return (a * (256 - f) + b * f) >> 8


LANE_MUL = (1, 40503, 22639, 51749)            # odd: a bijection of the pair index per lane
LANE_ADD = (0, 12345, 777, 31337)


def lane_pairs(idx, lanes):
    """(a, b) per byte lane of pair index idx (0..65535, any shape): lane L takes its own
    bijection of idx, so that each lane meets every pair."""
    a = np.zeros(idx.shape + (4,), np.int64)
    b = np.zeros_like(a)
    for L in lanes:
        k = (idx * LANE_MUL[L] + LANE_ADD[L]) & 0xffff
        a[..., L], b[..., L] = k >> 8, k & 255
    return a, b


H_DW, H_DH, H_RECTS = 257, 4096, 16             # 16 rectangles x 4096 rows = 65536 pairs per fraction


def h_domain(lanes):
    """Sources whose two rows of a pair are equal (2i, 2i+1) and whose render size is half their
    pixel size: the vertical merge is the identity and destination column x reads source
    columns (2x, 2x + 1) with fraction x - 1."""
    sw, sh = 2 * H_DW, 2 * H_DH
    xi = x_inc_of(sw, H_DW)
    x = np.arange(H_DW)
    sx, f = (x * xi) >> 16, ((x * xi) >> 8) & 255
    assert np.array_equal(sx, 2 * x) and sorted(set(f.tolist())) == list(range(256))
    rects = []
    for q in range(H_RECTS):
        y = np.arange(H_DH)[:, None]
        idx = (q * H_DH + y + x[None, :] * 977) & 0xffff       # bijective in y for every x
        a, b = lane_pairs(idx, lanes)
        src = np.zeros((H_DH, sw, 4), np.uint8)
        src[:, 0::2], src[:, 1::2] = a, b
        if 3 not in lanes:
            src[..., 3] = 255
        px = np.repeat(src, 2, axis=0)
        rects.append(dict(pixels=px, x=(q % 4) * H_DW, y=(q // 4) * H_DH, render_width=H_DW, render_height=H_DH))
    return rects, f


def decode_h(rects, f, lanes):
    """(a, b, f) per lane, read back from the source pixels and the row plan each rectangle gets."""
    keys = {L: [] for L in lanes}
    for r in rects:
        px = r["pixels"]
        plan = np.array(model_scale_rows(px.shape[0], r["render_height"]))
        assert np.array_equal(plan[:, 0], 2 * np.arange(plan.shape[0]))
        assert np.array_equal(px[plan[:, 0]], px[plan[:, 1]])     # the merge is the identity
        rows = px[plan[:, 0]].astype(np.int64)
        xi = x_inc_of(px.shape[1], r["render_width"])
        sx = (np.arange(r["render_width"]) * xi) >> 16
        for L in lanes:
            keys[L].append((rows[:, sx, L] << 16) | (rows[:, sx + 1, L] << 8) | f[None, :])
    return {L: distinct(np.concatenate([k.ravel() for k in ks])) for L, ks in keys.items()}


@pytest.mark.parametrize("lanes", [(0, 1, 2), (3,)], ids=["colour", "alpha"])
def test_scale_horizontal_every_input(ctx, lanes):
    """scale_mix_h: every (a, b, f), 2^24, on each byte lane; colour lanes at alpha 255, the
    alpha lane on its own (where it comes out 0 the pixel reads back as 0)."""
    rects, f = h_domain(lanes)
    cov = decode_h(rects, f, lanes)
    assert cov == {L: 1 << 24 for L in lanes}
    W, H = 4 * H_DW, (H_RECTS // 4) * H_DH
    got = readback_rects(ctx, 510, W, H, rects)
    for r in rects:
        px = r["pixels"][0::2].astype(np.int64)
        want = h_mix(px[:, 0::2], px[:, 1::2], f[None, :, None])
        x0, y0 = r["x"], r["y"]
        assert np.array_equal(got[y0:y0 + H_DH, x0:x0 + H_DW], visible(want)), (x0, y0)
    r = rects[0]
    assert np.array_equal(visible(model_scale(r["pixels"], H_DW, H_DH)), got[:H_DH, :H_DW])


V_DW, V_DH, V_RECTS = 4096, 257, 16


@pytest.mark.parametrize("lanes", [(0, 1, 2), (3,)], ids=["colour", "alpha"])
def test_scale_vertical_every_input(ctx, lanes):
    """The vertical merge a + (((b - a) * w + 128) >> 8): every (ca, cb, w) the row plan
    produces (weights 0..255 in the merge branch), columns paired so that the horizontal pass
    is the identity."""
    sw, sh = 2 * V_DW, 2 * V_DH
    plan = np.array(model_scale_rows(sh, V_DH))
    merge = plan[1:]
    assert plan[0].tolist() == [0, 0, 0]
    assert np.array_equal(merge[:, 0], 2 * np.arange(1, V_DH)) and np.array_equal(merge[:, 1], merge[:, 0] + 1)
    assert sorted(merge[:, 2].tolist()) == list(range(256))          # every weight once per column
    rects = []
    for q in range(V_RECTS):
        xcol = np.arange(V_DW)[None, :]
        j = np.arange(V_DH)[:, None]
        idx = (q * V_DW + xcol + j * 4099) & 0xffff                  # bijective in x for every row
        a, b = lane_pairs(idx, lanes)
        src = np.zeros((sh, V_DW, 4), np.uint8)
        src[0::2], src[1::2] = a, b
        if 3 not in lanes:
            src[..., 3] = 255
        px = np.repeat(src, 2, axis=1)
        rects.append(dict(pixels=px, x=0, y=q * V_DH, render_width=V_DW, render_height=V_DH))
    keys = {L: [] for L in lanes}
    for r in rects:
        px = r["pixels"].astype(np.int64)
        assert np.array_equal(px[:, 0::2], px[:, 1::2])               # the horizontal pass is the identity
        for L in lanes:
            ca, cb = px[merge[:, 0], 0::2, L], px[merge[:, 1], 0::2, L]
            keys[L].append((ca << 16) | (cb << 8) | merge[:, 2:3])
    assert {L: distinct(np.concatenate([k.ravel() for k in ks])) for L, ks in keys.items()} == \
        {L: 1 << 24 for L in lanes}
    got = readback_rects(ctx, 511, V_DW, V_RECTS * V_DH, rects)
    for r in rects:
        px = r["pixels"][:, 0::2].astype(np.int64)
        ca, cb = px[plan[:, 0]], px[plan[:, 1]]
        want = ca + (((cb - ca) * plan[:, 2][:, None, None] + 128) >> 8)
        assert np.array_equal(got[r["y"]:r["y"] + V_DH], visible(want)), r["y"]
    r = rects[1]
    assert np.array_equal(visible(model_scale(r["pixels"], V_DW, V_DH)), got[V_DH:2 * V_DH])


def test_scale_every_small_geometry(ctx):
    """Every source width 2..40 x render width 1..80 (source heights 2..5, render heights
    1..6), 64 rectangles per install, against helpers.model_scale through model_blend."""
    specs = [(sw, rw) for sw in range(2, 41) for rw in range(1, 81)]
    W, cell = 80, 8
    n = 0
    for start in range(0, len(specs), 64):
        part = specs[start:start + 64]
        rects = []
        for k, (sw, rw) in enumerate(part):
            i = start + k
            sh, rh = 2 + i % 4, 1 + (i * 7) % 6
            rects.append(dict(pixels=random_overlay(sw, sh, i, premultiplied=bool(i & 1), density=0.9),
                              x=0, y=k * cell, render_width=rw, render_height=rh, premultiplied=True))
            n += 1
        H = len(part) * cell
        assert np.array_equal(readback_rects(ctx, 512, W, H, rects), model_readback(W, H, rects)), start
    assert n == 39 * 80


def test_scale_clipped_one_pixel_and_largest_sides(ctx):
    """Scaled rectangles hanging over every frame edge, scaled down to 1x1, and sources of
    32768 x 2 and 2 x 32768 -- the largest side accepted -- scaled to small sizes."""
    r = np.random.default_rng(5)
    W, H = 120, 90
    rects = [dict(pixels=random_overlay(37, 23, 1), x=-11, y=-7, render_width=50, render_height=30),
             dict(pixels=random_overlay(19, 41, 2), x=100, y=-3, render_width=31, render_height=17),
             dict(pixels=random_overlay(64, 9, 3), x=-20, y=75, render_width=45, render_height=33),
             dict(pixels=random_overlay(5, 5, 4), x=110, y=80, render_width=29, render_height=27),
             dict(pixels=random_overlay(40, 30, 5), x=60, y=40, render_width=1, render_height=1),
             dict(pixels=random_overlay(2, 2, 6), x=62, y=40, render_width=1, render_height=1)]
    for rc in rects[4:]:
        rc["pixels"][..., 3] = np.maximum(rc["pixels"][..., 3], 1)     # the single pixel shows
    want = model_readback(W, H, rects)
    assert np.array_equal(want, oracle_blend("BGRA", W, H, [np.zeros((H, 4 * W), np.uint8)], rects,
                                             True)[0].reshape(H, W, 4))
    assert np.array_equal(readback_rects(ctx, 513, W, H, rects), want)
    for sw, sh, rw, rh in ((32768, 2, 100, 3), (2, 32768, 3, 100), (32768, 3, 77, 1), (3, 32768, 1, 61)):
        px = r.integers(0, 256, (sh, sw, 4), dtype=np.uint8)
        px[..., 3] = np.maximum(px[..., 3], 1)
        rl = [dict(pixels=px, x=1, y=2, render_width=rw, render_height=rh)]
        want = model_readback(rw + 2, rh + 3, rl)
        assert np.array_equal(want[2:2 + rh, 1:1 + rw], visible(model_scale(px, rw, rh)))
        assert np.array_equal(readback_rects(ctx, 514, rw + 2, rh + 3, rl), want), (sw, sh)


@pytest.mark.parametrize("sw,sh,rw,rh", [
    (32769, 2, 100, 2), (2, 32769, 2, 100),         # source side
    (32769, 3, 0, 5), (3, 32769, 5, 0),             # effective render side (0: the pixel size)
    (4, 4, 32769, 4), (4, 4, 4, 32769),             # render side
])
def test_scale_refuses_sides_above_32768(ctx, sw, sh, rw, rh):
    """Above 32768 on a side the scaler's 32-bit 16.16 positions overflow: refused with
    INVALID_ARGUMENT before any work -- no counter moves -- and the stream keeps its overlay."""
    before_px = random_overlay(6, 5, 9)
    prev = [dict(pixels=before_px, x=3, y=2)]
    ctx.overlay_set_rectangles(515, prev)
    big = np.full((sh, sw, 4), 200, np.uint8)
    st = ctx.stats()
    with pytest.raises(tbm.TtmlBlendError) as e:
        ctx.overlay_set_rectangles(515, [dict(pixels=big, x=0, y=0, render_width=rw, render_height=rh)])
    assert e.value.code == tbm.ERROR_INVALID_ARGUMENT
    assert ctx.stats() == st
    assert np.array_equal(run_bgra(ctx, 515, 12, 9), model_readback(12, 9, prev))


def test_unscaled_rectangle_keeps_its_limits(ctx):
    """The limit is the scaler's: a 32769-pixel side at its own render size is accepted."""
    px = np.zeros((2, 32769, 4), np.uint8)
    px[1, 5] = (1, 2, 3, 255)
    ctx.overlay_set_rectangles(516, [dict(pixels=px, x=0, y=0)])
    got = run_bgra(ctx, 516, 8, 2)
    assert got[1, 5].tolist() == [1, 2, 3, 255] and np.count_nonzero(got) == 4


# ---------------------------------------------------------------------------
# R: region composition (pixman 8-bit OVER / IN, Cairo's colour conversion)

def mul_un8(a, b):
    """a * b / 255 rounded to nearest: a * b / 255 is never half-way for bytes."""
    return (2 * a * b + 255) // 510


def over_un8(s, sa, d):
    return np.minimum(s + mul_un8(d, 255 - sa), 255)


def cairo_pixel(rgba):
    """_cairo_color_compute_shorts then >> 8: (B, G, R, A) bytes of a 0xRRGGBBAA colour."""
    r, g, b, a = [((rgba >> s) & 255) / 255.0 for s in (24, 16, 8, 0)]
    short = lambda v: (int(v * 65535.0 + 0.5) & 0xffff) >> 8
    return short(b * a), short(g * a), short(r * a), short(a)


def m8_of(op):
    return 255 if op >= 1.0 else (int(op * 65535.0 + 0.5) & 0xffff) >> 8


def test_pixman_models_agree():
    """The restatements above against pixman's own formula ((t >> 8) + t) >> 8, t = a*b + 0x80."""
    a, b = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    t = a * b + 0x80
    assert np.array_equal(mul_un8(a, b), ((t >> 8) + t) >> 8)


def readback_regions(ctx, stream, w, h, regions):
    ctx.overlay_set_regions(stream, w, h, regions)
    return run_bgra(ctx, stream, w, h)


def test_region_over_every_input(ctx):
    """Two layered regions on one box, the first layer opaque (its colours are d_c), the second
    any (s_c, s_a): every (s_c, s_a, d_c) on each colour channel, s_c > s_a (a layer that is not
    premultiplied, where min (., 255) saturates) included."""
    W = H = 4096
    t = np.arange(W * H, dtype=np.int64).reshape(H, W)
    sa, u = t >> 16, t & 0xffff
    top = np.zeros((H, W, 4), np.uint8)
    bottom = np.zeros((H, W, 4), np.uint8)
    top[..., 3], bottom[..., 3] = sa, 255
    for ch in range(3):
        k = (u * LANE_MUL[ch + 1] + LANE_ADD[ch + 1]) & 0xffff
        top[..., ch], bottom[..., ch] = k >> 8, k & 255
    sa_i = top[..., 3].astype(np.int64)
    for ch in range(3):
        key = (top[..., ch].astype(np.int64) << 16) | (sa_i << 8) | bottom[..., ch]
        assert distinct(key) == 1 << 24, ch
    assert (top[..., :3] > top[..., 3:]).any()
    regions = [dict(x=0, y=0, w=W, h=H, layer=bottom), dict(x=0, y=0, w=W, h=H, layer=top)]
    want = np.empty((H, W, 4), np.uint8)
    s, d = top.astype(np.int64), bottom.astype(np.int64)
    for ch in range(4):
        want[..., ch] = over_un8(s[..., ch], sa_i, d[..., ch])
    assert (want[..., 3] == 255).all()
    crop = [dict(r, h=64, layer=np.ascontiguousarray(r["layer"][:64])) for r in regions]
    assert np.array_equal(oracle.compose_regions(crop, W, 64), want[:64])
    assert np.array_equal(readback_regions(ctx, 520, W, H, regions), want)


def m8_ends():
    """For every m8 = (uint16) (op * 65535 + 0.5) >> 8 (op < 1): the smallest and the largest
    double opacity that gives it."""
    ends = []
    for k in range(256):
        lo = max(0.0, (256 * k - 0.5) / 65535.0)
        while lo > 0.0 and m8_of(math.nextafter(lo, -1.0)) == k:
            lo = math.nextafter(lo, -1.0)
        while m8_of(lo) < k:
            lo = math.nextafter(lo, 2.0)
        hi = min(math.nextafter(1.0, 0.0), (256 * k + 255.5) / 65535.0)
        while m8_of(hi) > k:
            hi = math.nextafter(hi, -1.0)
        while hi < math.nextafter(1.0, 0.0) and m8_of(math.nextafter(hi, 2.0)) == k:
            hi = math.nextafter(hi, 2.0)
        assert m8_of(lo) == k == m8_of(hi) and lo < 1.0 and hi < 1.0
        ends += [lo, hi]
    return ends


def test_region_opacity_every_group_input(ctx):
    """cairo_paint_with_alpha of the group: every (g_c, m8) through in_un8x4, with opacities at
    both ends of every m8 step (512 regions of 16 x 16, 64 per install)."""
    ops = m8_ends()
    assert sorted({m8_of(o) for o in ops}) == list(range(256)) and len(ops) == 512
    p = np.arange(256)
    layer = np.zeros((16, 16, 4), np.uint8)
    layer[..., 0] = p.reshape(16, 16)
    layer[..., 1] = ((p + 85) & 255).reshape(16, 16)
    layer[..., 2] = ((p * 3 + 170) & 255).reshape(16, 16)
    layer[..., 3] = 255
    seen = set()
    for start in range(0, len(ops), 64):
        part = ops[start:start + 64]
        regions = [dict(x=16 * (k % 8), y=16 * (k // 8), w=16, h=16, opacity=op, layer=layer)
                   for k, op in enumerate(part)]
        want = np.zeros((128, 128, 4), np.uint8)
        for k, op in enumerate(part):
            m = m8_of(op)
            want[16 * (k // 8):16 * (k // 8) + 16, 16 * (k % 8):16 * (k % 8) + 16] = mul_un8(layer.astype(np.int64), m)
            for ch in range(3):
                seen.update((int(g), m) for g in layer[..., ch].ravel())
        assert np.array_equal(oracle.compose_regions(regions, 128, 128), want)
        assert np.array_equal(readback_regions(ctx, 521, 128, 128, regions), visible(want)), start
    assert len(seen) == 1 << 16


def test_region_background_every_colour(ctx):
    """cairo_solid_pixel for every (c, a): 256 alphas x 86 regions, R, G and B each a colour."""
    cells = []
    for a in range(256):
        for j in range(86):
            c = [(3 * j + i) % 256 for i in range(3)]
            cells.append((c[0] << 24) | (c[1] << 16) | (c[2] << 8) | a)
    seen = {(((v >> s) & 255), v & 255) for v in cells for s in (24, 16, 8)}
    assert len(seen) == 1 << 16
    for start in range(0, len(cells), 64):
        part = cells[start:start + 64]
        regions = [dict(x=4 * (k % 8), y=4 * (k // 8), w=4, h=4, background_color=v, opacity=1.0)
                   for k, v in enumerate(part)]
        want = np.zeros((32, 32, 4), np.uint8)
        for k, v in enumerate(part):
            want[4 * (k // 8):4 * (k // 8) + 4, 4 * (k % 8):4 * (k % 8) + 4] = cairo_pixel(v) if v else 0
        assert np.array_equal(oracle.compose_regions(regions, 32, 32), want)
        assert np.array_equal(readback_regions(ctx, 522, 32, 32, regions), visible(want)), start


def text_layer(w, h, seed):
    px = random_overlay(w, h, seed, premultiplied=True, density=0.8)
    px[(np.arange(h)[:, None] + np.arange(w)[None, :]) % 5 == 0] = 0
    return px


@pytest.mark.parametrize("edge", ["left", "top", "right", "bottom", "all"])
def test_region_layers_over_the_frame_edges(ctx, edge):
    """Text layers on regions that hang over a frame edge: the kernel reads the layer from
    (p.lx, p.ly) on, against oracle.compose_regions."""
    W, H = 96, 64
    box = {"left": (-13, 10, 50, 30), "top": (20, -9, 40, 33), "right": (70, 8, 41, 27),
           "bottom": (15, 45, 44, 31), "all": (-7, -5, 110, 75)}[edge]
    x, y, w, h = box
    regions = [dict(x=x, y=y, w=w, h=h, background_color=0x20406080, opacity=1.0, layer=text_layer(w, h, 1)),
               dict(x=x + 3, y=y + 2, w=w, h=h, background_color=0, opacity=0.7, layer=text_layer(w, h, 2)),
               dict(x=x - 2, y=y + 4, w=w, h=h, background_color=0xC0A000FF, opacity=0.35, layer=text_layer(w, h, 3))]
    want = oracle.compose_regions(regions, W, H)
    assert np.count_nonzero(want[..., 3]) > W * H // 8                # the layers are really there
    assert np.array_equal(readback_regions(ctx, 523, W, H, regions), visible(want))


# ---------------------------------------------------------------------------
# B: the outline blur

BLUR_TILE = (32, 8)


def blur_smem(r):
    """launch_blur's dynamic shared memory: the tile with its halo, and the taps."""
    return ((BLUR_TILE[0] + 2 * r) * (BLUR_TILE[1] + 2 * r) + (2 * r + 1) ** 2) * 4


def gauss_taps(r, sigma):
    """gst_ttml_blur_create_gaussian_kernel restated: normalised exp (-(x^2 + y^2) / 2 sigma^2)
    in 16.16 fixed point, summed in the reference's order."""
    s2 = 2.0 * sigma * sigma
    s1 = 1.0 / (math.pi * s2)
    tmp = [s1 * math.exp(-(float(x * x) + float(y * y)) / s2) for x in range(-r, r + 1) for y in range(-r, r + 1)]
    total = 0.0
    for v in tmp:
        total += v
    return np.array([int((v / total) * 65536.0) for v in tmp], np.int64).reshape(2 * r + 1, 2 * r + 1)


def conv_model(img, taps):
    """Pixels outside the image are transparent; CLIP ((sum + 0x8000) >> 16) per channel."""
    r = taps.shape[0] // 2
    h, w = img.shape[:2]
    pad = np.zeros((h + 2 * r, w + 2 * r, 4), np.int64)
    pad[r:r + h, r:r + w] = img
    acc = np.zeros((h, w, 4), np.int64)
    for i in range(2 * r + 1):
        win = np.lib.stride_tricks.sliding_window_view(pad[i:i + h], 2 * r + 1, axis=1)[:, :w]
        acc += np.einsum("hwcj,j->hwc", win, taps[i])
    return np.clip((acc + 0x8000) >> 16, 0, 255).astype(np.uint8)


def blur_api(ctx, img, r, sigma, dst_pad=0, inplace=False):
    """fluc_ttmlblend_blur_argb32 with the caller's strides; the destination's row padding must
    stay untouched."""
    h, w = img.shape[:2]
    if inplace:
        dst = img
    else:
        buf = np.full((h, w + dst_pad, 4), 0xA5, np.uint8)
        dst = buf[:, :w]
    rc = ctx.lib.fluc_ttmlblend_blur_argb32(ctx.h, img.ctypes.data, w, h, img.strides[0], r, float(sigma),
                                            dst.ctypes.data, dst.strides[0])
    assert rc == 0, f"blur_argb32 returned {rc} at radius {r}"
    if not inplace and dst_pad:
        assert (buf[:, w:] == 0xA5).all()
    return np.array(dst)


def padded(img, pad):
    h, w = img.shape[:2]
    buf = np.zeros((h, w + pad, 4), np.uint8)
    buf[:, :w] = img
    return buf[:, :w]


def test_gauss_taps_restated():
    for r in (0, 1, 7, 33, 34, 64):
        assert np.array_equal(gauss_taps(r, 0.5 + r / 3), oracle.gaussian_kernel(r, 0.5 + r / 3)), r


BLUR_SHAPES = [(5, 3, 0, 0), (33, 9, 3, 5), (17, 13, 1, 0), (1, 1, 0, 2)]     # w, h, src pad px, dst pad px


def test_blur_every_radius(ctx):
    """Every radius 0..64 on small odd shapes (w and h below 2r + 1, one pixel wider and
    taller than a 32 x 8 tile, a single pixel) with padded source and destination strides,
    against the oracle, and against the numpy convolution on one shape. The 48 KB dynamic
    shared-memory boundary of launch_blur lies between radius 33 and 34."""
    big = [r for r in range(65) if blur_smem(r) > 48 * 1024]
    assert big[0] == 34 and blur_smem(33) <= 48 * 1024 and blur_smem(64) <= 200 * 1024
    for r in range(65):
        sigma = 0.5 + r / 3
        taps = gauss_taps(r, sigma)
        for k, (w, h, sp, dp) in enumerate(BLUR_SHAPES):
            img = padded(random_overlay(w, h, 1000 * k + r, premultiplied=True, density=0.6), sp)
            got = blur_api(ctx, img, r, sigma, dp)
            assert np.array_equal(got, oracle.blur_argb32(img, r, sigma)), (r, w, h)
            if k == 2 or r in (33, 34):
                assert np.array_equal(got, conv_model(img, taps)), (r, w, h)


@pytest.mark.parametrize("r", [1, 7, 33, 34, 64])
def test_blur_impulses_every_value_and_tap(ctx, r):
    """Impulses of every value v in 0..255 (64 pixels x 4 channels), (2r + 1) apart: around each
    one the output is clamp ((v * tap + 0x8000) >> 16) for every tap, and 0 between them."""
    sigma = r / 2
    taps = gauss_taps(r, sigma)
    s = 2 * r + 1
    img = np.zeros((8 * s, 8 * s, 4), np.uint8)
    want = np.zeros((8 * s, 8 * s, 4), np.int64)
    pairs = set()
    for k in range(64):
        cy, cx = (k // 8) * s, (k % 8) * s
        v = 4 * k + np.arange(4)
        img[cy + r, cx + r] = v
        want[cy:cy + s, cx:cx + s] = np.minimum((v[None, None, :] * taps[:, :, None] + 0x8000) >> 16, 255)
        pairs.update((int(x), t) for x in v for t in range(s * s))
    assert len(pairs) == 256 * s * s
    assert sorted(img[r::s, r::s].ravel().tolist()) == list(range(256))
    assert np.array_equal(blur_api(ctx, img, r, sigma), want.astype(np.uint8))


def test_blur_in_place(ctx):
    """dst == src through the API (the library stages through device buffers)."""
    for r, (w, h) in ((5, (37, 11)), (40, (45, 19))):
        img = random_overlay(w, h, 77 + r, premultiplied=True, density=0.6)
        want = oracle.blur_argb32(img, r, r / 2)
        work = img.copy()
        assert np.array_equal(blur_api(ctx, work, r, r / 2, inplace=True), want)
        assert np.array_equal(work, want)


# ---------------------------------------------------------------------------
# W: row spans, the crop, and the lazy / opaque-skip decisions

def span_rows(W, cols):
    """One rectangle row per column c: c and W - 1 - c visible (the row's first and last)."""
    px = np.zeros((len(cols), 1, W, 4), np.uint8)
    for i, c in enumerate(cols):
        px[i, 0, c] = (c & 255, (c >> 8) & 255, 7, 255)
        px[i, 0, W - 1 - c] = (c & 255, 99, (c >> 8) & 255, 200)
    return px


def check_columns(ctx, W, cols):
    for start in range(0, len(cols), 64):
        part = cols[start:start + 64]
        px = span_rows(W, part)
        rects = [dict(pixels=px[i], x=0, y=i) for i in range(len(part))]
        got = readback_rects(ctx, 530, W, len(part), rects)
        assert np.array_equal(got, px[:, 0]), (W, part[0])


def test_crop_keeps_a_pixel_at_every_column(ctx):
    """Rows with one visible pixel at c and one at W - 1 - c, for every c of every width
    1..300: the row-span reduction over warps and the 128-thread block keeps both."""
    for W in range(1, 301):
        cols = list(range((W + 1) // 2))
        assert sorted(set(cols) | {W - 1 - c for c in cols}) == list(range(W))
        check_columns(ctx, W, cols)


@pytest.mark.parametrize("W", [4096, 32768])
def test_crop_keeps_a_pixel_at_every_column_wide(ctx, W):
    check_columns(ctx, W, list(range(W // 2)))


def model_groups(img):
    """ttmlblend_rowspan_kernel restated: per row the span (first, last) of alpha != 0 and the
    16-pixel groups (aligned to the rectangle) with any alpha / all alpha 255."""
    a = img[..., 3].astype(np.int64)
    h, w = a.shape
    g = -(-w // 16)
    pad = np.zeros((h, 16 * g), np.int64)
    pad[:, :w] = a
    grp = pad.reshape(h, g, 16)
    on = (grp != 0).any(2).sum(1)
    full = np.zeros((h, 16 * g), bool)
    full[:, :w] = a == 255
    opq = full.reshape(h, g, 16).all(2).sum(1)
    spans = []
    for y in range(h):
        nz = np.flatnonzero(a[y])
        spans.append((int(nz[0]), int(nz[-1])) if nz.size else (w, -1))
    return spans, on, opq


def model_crop(spans, min_gap=16, max_runs=8):
    """crop_runs restated: row runs closer than min_gap merge; then the closest pair, until
    max_runs remain. Returns (x, y, w, h) sub-rectangles."""
    runs = []
    for y, (x0, x1) in enumerate(spans):
        if x1 < x0:
            continue
        if runs and y - runs[-1][1] < min_gap:
            r = runs[-1]
            runs[-1] = [r[0], y + 1, min(r[2], x0), max(r[3], x1 + 1)]
        else:
            runs.append([y, y + 1, x0, x1 + 1])
    while len(runs) > max_runs:
        best = 0
        for i in range(1, len(runs) - 1):
            if runs[i + 1][0] - runs[i][1] < runs[best + 1][0] - runs[best][1]:
                best = i
        a, b = runs[best], runs.pop(best + 1)
        runs[best] = [a[0], b[1], min(a[2], b[2]), max(a[3], b[3])]
    return [(r[2], r[0], r[3] - r[2], r[1] - r[0]) for r in runs]


def model_decisions(img):
    """(lazy in place, opaque skip) of one rectangle at global alpha 1: decide_lazy restated."""
    spans, on, opq = model_groups(img)
    g_all = g_on = g_opq = 0
    for (x, y, w, h) in model_crop(spans):
        g_all += -(-w // 16) * h
        g_on += int(on[y:y + h].sum())
        g_opq += int(opq[y:y + h].sum())
    tf = 1.0 - g_on / g_all if g_all else 0.0
    of = g_opq / g_all if g_all else 0.0
    return tf + of >= 0.3, of >= 0.3


def group_image(W, H, x0, x1, n_opaque, n_empty):
    """Rows visible from x0 to x1 - 1; inside, whole 16-pixel groups (aligned to the rectangle)
    made opaque or left empty, n of each in row-major order; the rest of a row has alpha 1..254."""
    img = np.zeros((H, W, 4), np.uint8)
    img[:, x0:x1] = (10, 20, 30, 128)
    inner = [g for g in range(W // 16) if 16 * g > x0 and 16 * g + 16 < x1]
    slots = [(y, g) for y in range(H) for g in inner]
    assert n_opaque + n_empty <= len(slots)
    for y, g in slots[:n_opaque]:
        img[y, 16 * g:16 * g + 16] = (1, 2, 3, 255)
    for y, g in slots[n_opaque:n_opaque + n_empty]:
        img[y, 16 * g:16 * g + 16] = 0
    return img


def flip(make, which):
    """The n at which decision `which` turns on, and the images at n - 1 and n."""
    prev = None
    for n in range(0, 400):
        d = model_decisions(make(n))[which]
        if prev is False and d:
            return n
        prev = d
    raise AssertionError("no flip")


@pytest.mark.skipif(any(k in os.environ for k in LAZY_KNOBS), reason="a knob forces the paths")
@pytest.mark.parametrize("geom", [(160, 16, 0, 160), (200, 20, 8, 158)], ids=["aligned", "cropped"])
@pytest.mark.parametrize("which", ["opaque", "transparent", "mixed"])
def test_lazy_and_opaque_skip_flip_at_the_threshold(ctx, geom, which):
    """The figures decide_lazy compares with 0.3, from the group counts of the cropped
    sub-rectangles: one group either side of the flip, in place (lazy_launches) and out of
    place (opaque_skip_launches)."""
    W, H, x0, x1 = geom
    if which == "opaque":
        make, idx = (lambda n: group_image(W, H, x0, x1, n, 0)), 1
    elif which == "transparent":
        make, idx = (lambda n: group_image(W, H, x0, x1, 0, n)), 0
    else:
        make, idx = (lambda n: group_image(W, H, x0, x1, 12, n)), 0
    n = flip(make, idx)
    for img in (make(n - 1), make(n)):
        lazy, skip = model_decisions(img)
        ctx.overlay_set_rectangles(531, [dict(pixels=img, x=0, y=0)])
        for inplace in (False, True):
            st = ctx.stats()
            got = run_bgra(ctx, 531, W, H, inplace=inplace)
            d = {k: v - st[k] for k, v in ctx.stats().items()}
            assert np.array_equal(got, visible(img))
            assert d["group_launches"] + d["multi_launches"] == 1, d
            if inplace:
                assert d["lazy_launches"] == int(lazy) and d["opaque_skip_launches"] == 0, (n, d)
            else:
                assert d["opaque_skip_launches"] == int(skip) and d["lazy_launches"] == 0, (n, d)
    assert model_decisions(make(n - 1))[idx] is False and model_decisions(make(n))[idx] is True


# ---------------------------------------------------------------------------
# C: averaged chroma (set_chroma_mode(True))

@pytest.fixture
def avg_ctx(ctx):
    ctx.set_chroma_mode(True)
    try:
        yield ctx
    finally:
        ctx.set_chroma_mode(False)


FMT_420 = ("I420", "YV12", "NV12", "NV21")


def avg_cases(W, H):
    """One rectangle per case: every origin parity x every width / height parity inside the
    frame, then clipped on each edge and on all four."""
    out = [(x, y, w, h) for x in (4, 5) for y in (2, 3) for w in (6, 7) for h in (4, 5)]
    out += [(-3, 4, 9, 6), (5, -3, 7, 8), (W - 5, 3, 9, 7), (4, H - 3, 8, 7), (-1, -2, W + 3, H + 5)]
    return out


@pytest.mark.parametrize("fmt", FMT_420)
@pytest.mark.parametrize("W,H", [(37, 23), (38, 24)])
def test_chroma_average_parities_and_clips(avg_ctx, fmt, W, H):
    cases = avg_cases(W, H)
    assert {(x & 1, y & 1, w & 1, h & 1) for x, y, w, h in cases[:16]} == \
        {(a, b, c, d) for a in (0, 1) for b in (0, 1) for c in (0, 1) for d in (0, 1)}
    for i, (x, y, w, h) in enumerate(cases):
        px = random_overlay(w, h, 50 + i, premultiplied=bool(i & 1), density=0.8)
        rl = [dict(pixels=px, x=x, y=y, premultiplied=bool(i & 1))]
        planes = random_frame(fmt, W, H, i)
        want = model_blend(fmt, W, H, copy_planes(planes), rl, chroma_average=True)
        avg_ctx.overlay_set_rectangles(540, rl)
        assert_planes_equal(run_fmt(avg_ctx, 540, fmt, W, H, planes), want, f"{fmt} {W}x{H} {(x, y, w, h)}")


@pytest.mark.parametrize("fmt", FMT_420)
def test_chroma_average_spans_across_blocks(avg_ctx, fmt):
    """Spans of more than 512 luma columns: a chroma row crosses 256-thread blocks."""
    W, H = 1400, 20
    for i, (x, w) in enumerate(((0, 1400), (1, 1031), (7, 514), (300, 1099))):
        px = random_overlay(w, 15, 70 + i, premultiplied=True, density=0.85)
        rl = [dict(pixels=px, x=x, y=i % 2 + 1)]
        planes = random_frame(fmt, W, H, 90 + i)
        want = model_blend(fmt, W, H, copy_planes(planes), rl, chroma_average=True)
        avg_ctx.overlay_set_rectangles(541, rl)
        assert_planes_equal(run_fmt(avg_ctx, 541, fmt, W, H, planes), want, f"{fmt} x={x} w={w}")


# ---------------------------------------------------------------------------
# X: fades of what the per-cue kernels made

@pytest.mark.parametrize("fmt", ["I420", "NV12", "BGRA"])
def test_fade_of_a_scaled_rectangle_installed_below_one(ctx, fmt):
    """The first overlay_set_global_alpha of a scaled rectangle installed at 0.6 prepares again
    from the resident scaled pixels; every frame equals the oracle at the value of its time."""
    W, H = 96, 64
    base = dict(pixels=random_overlay(30, 20, 3, premultiplied=False), x=-5, y=7, render_width=71,
                render_height=45, premultiplied=False)
    other = dict(pixels=random_overlay(20, 12, 4), x=50, y=30)
    planes = random_frame(fmt, W, H, 12)
    ctx.overlay_set_rectangles(550, [dict(base, global_alpha=0.6), other])
    want = oracle_blend(fmt, W, H, copy_planes(planes), [dict(base, global_alpha=0.6), other])
    assert_planes_equal(run_fmt(ctx, 550, fmt, W, H, planes), want, "installed at 0.6")
    for ga in (0.3, 1.0, 0.85):
        ctx.overlay_set_global_alpha(550, [ga, 1.0])
        want = oracle_blend(fmt, W, H, copy_planes(planes), [dict(base, global_alpha=ga), other])
        assert_planes_equal(run_fmt(ctx, 550, fmt, W, H, planes), want, f"faded to {ga}")


@pytest.mark.parametrize("fmt", ["I420", "NV12", "BGRA"])
def test_fade_of_a_region_form_overlay(ctx, fmt):
    W, H = 96, 64
    regions = [dict(x=-6, y=4, w=50, h=20, background_color=0x10204080, opacity=0.8, layer=text_layer(50, 20, 5)),
               dict(x=40, y=30, w=70, h=40, background_color=0xFFFFFFFF, opacity=1.0, layer=text_layer(70, 40, 6))]
    ov = oracle.compose_regions(regions, W, H)
    planes = random_frame(fmt, W, H, 13)
    ctx.overlay_set_regions(551, W, H, regions)
    for ga in (1.0, 0.4, 0.75):
        if ga != 1.0:
            ctx.overlay_set_global_alpha(551, ga)
        want = oracle_blend(fmt, W, H, copy_planes(planes), [dict(pixels=ov, x=0, y=0, global_alpha=ga)])
        assert_planes_equal(run_fmt(ctx, 551, fmt, W, H, planes), want, f"regions at {ga}")
