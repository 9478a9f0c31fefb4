"""CPU tests of the oracle (oracle/ttmlblend_ref.c): known answers from the published
BT.709 8-bit matrix and OVER formulas, agreement with an independent numpy model of the
net per-plane semantics, and the frozen golden fixtures. PARITY UNPINNED: the reference
holds no vector for this path (SURVEY.md section 8c), so the fixtures are oracle-generated
and only the known-answer tests come from outside the oracle."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from helpers import (ALL_FORMATS, PACKED, PACKED_ORDER, PLANAR_420, copy_planes, model_blend,
                     oracle_blend, random_frame, random_overlay, wl)
from oracle import oracle

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_div255_magic_is_exact():
    """(x * 32897) >> 23 == x / 255 on every numerator the kernels can form (<= 255*255)."""
    x = np.arange(0, 66299, dtype=np.uint64)
    assert np.array_equal((x * 32897) >> 23, x // 255)
    assert ((66299 * 32897) >> 23) != 66299 // 255      # and the bound is tight
    # the two-lane form the kernels use: (x + 1 + (x >> 8)) >> 8, exact up to 65534
    x = np.arange(0, 65535, dtype=np.uint64)
    assert np.array_equal((x + 1 + (x >> 8)) >> 8, x // 255)
    assert ((65535 + 1 + (65535 >> 8)) >> 8) != 65535 // 255
    # two lanes in one 32-bit register never carry into each other (lanes <= 255*255)
    lo, hi = np.meshgrid(np.array([0, 1, 254, 255, 65024, 65025], dtype=np.uint64),
                         np.array([0, 1, 254, 255, 65024, 65025], dtype=np.uint64))
    e = (lo | (hi << 16)) & 0xFFFFFFFF
    t = (e + ((e >> 8) & 0x00FF00FF) + 0x00010001) & 0xFFFFFFFF
    assert np.array_equal((t >> 8) & 0xFF, lo // 255) and np.array_equal((t >> 24) & 0xFF, hi // 255)


def test_magic_row_division_is_exact():
    """umulhi(item, ceil(2^32/nv)) == item / nv for every window the host accepts."""
    for nv in (1, 2, 3, 5, 7, 80, 120, 240, 241, 480, 960, 1023, 2048):
        if nv == 1:
            continue
        magic = ((1 << 32) + nv - 1) // nv
        e = magic * nv - (1 << 32)
        max_items = ((1 << 32) - 1) // e if e else 1 << 31
        max_items = min(max_items, 1 << 31)
        probe = np.unique(np.concatenate([
            np.arange(0, min(max_items, 200000)),
            np.arange(max(0, max_items - 200000), max_items),
            (np.arange(1, 4000) * nv) - 1, np.arange(1, 4000) * nv])).astype(np.uint64)
        probe = probe[probe < max_items]
        assert np.array_equal((probe * np.uint64(magic)) >> np.uint64(32), probe // np.uint64(nv)), nv


@pytest.mark.parametrize("rgb,yuv", [
    ((255, 255, 255), (235, 127, 128)),     # white  -> Y 235; U row sums to -1 => 127
    ((0, 0, 0), (16, 128, 128)),            # black  -> Y 16
    ((255, 0, 0), (62, 102, 239)),          # red    (BT.709: 63 / 102 / 240 before truncation)
    ((0, 255, 0), (172, 41, 26)),           # green
    ((0, 0, 255), (31, 239, 118)),          # blue
])
def test_matrix_known_answers(oracle_lib, rgb, yuv):
    line = np.array([255, *rgb], dtype=np.uint8)
    oracle_lib.tbref_matrix_rgb_to_yuv(line.ctypes.data, 1)
    assert tuple(line[1:]) == yuv
    # premultiplied at alpha 128: un-premultiply must give the same colour back
    a = 128
    pre = np.array([a, *[(c * a + 127) // 255 for c in rgb]], dtype=np.uint8)
    oracle_lib.tbref_matrix_prea_rgb_to_yuv(pre.ctypes.data, 1)
    assert pre[0] == a and tuple(pre[1:]) == yuv


def test_matrix_yuv_to_rgb_known_answers(oracle_lib):
    for yuv, rgb in (((235, 128, 128), (254, 254, 255)), ((16, 128, 128), (0, 0, 0))):
        line = np.array([255, *yuv], dtype=np.uint8)
        oracle_lib.tbref_matrix_yuv_to_rgb(line.ctypes.data, 1)
        assert tuple(line[1:]) == rgb


def _one_px_overlay(b, g, r, a):
    return np.array([[[b, g, r, a]]], dtype=np.uint8)


def test_opaque_white_pixel_on_i420():
    """a=255 white at an even/even position replaces Y and the sited chroma sample."""
    planes = [np.full((4, 4), 50, np.uint8), np.full((2, 2), 60, np.uint8), np.full((2, 2), 70, np.uint8)]
    oracle_blend("I420", 4, 4, planes, [dict(pixels=_one_px_overlay(255, 255, 255, 255), x=2, y=2)])
    assert planes[0][2, 2] == 235 and (planes[0] == 50).sum() == 15
    assert planes[1][1, 1] == 127 and planes[2][1, 1] == 128
    assert (planes[1] == 60).sum() == 3 and (planes[2] == 70).sum() == 3


def test_chroma_is_point_sampled_not_averaged():
    """A pixel at odd x or odd y changes luma only: pack_I420/NV12 write chroma on even lines
    from the even pixel of each pair (SURVEY.md finding 4)."""
    for (x, y) in ((1, 0), (0, 1), (3, 3)):
        for fmt in ("I420", "NV12"):
            planes = random_frame(fmt, 6, 6, 3)
            before = copy_planes(planes)
            oracle_blend(fmt, 6, 6, planes, [dict(pixels=_one_px_overlay(10, 200, 30, 255), x=x, y=y)])
            for p, q in zip(planes[1:], before[1:]):
                assert np.array_equal(p, q)
            assert (planes[0] != before[0]).sum() <= 1


def test_half_alpha_known_answer_bgra():
    """Premultiplied source on an opaque BGRA frame: out = Cs + Cd*(255-a)/255, alpha 255."""
    frame = np.array([[10, 20, 30, 255]], dtype=np.uint8)          # B,G,R,A
    ov = _one_px_overlay(64, 32, 100, 128)
    oracle_blend("BGRA", 1, 1, [frame], [dict(pixels=ov, x=0, y=0)])
    assert list(frame[0]) == [64 + 10 * 127 // 255, 32 + 20 * 127 // 255, 100 + 30 * 127 // 255, 255]


def test_straight_alpha_known_answer_ayuv():
    frame = np.array([[255, 100, 110, 120]], dtype=np.uint8)       # A,Y,U,V
    ov = _one_px_overlay(255, 255, 255, 128)                        # straight white, a=128
    oracle_blend("AYUV", 1, 1, [frame], [dict(pixels=ov, x=0, y=0, premultiplied=False)])
    want = [255] + [(s * 128 + d * 127) // 255 for s, d in ((235, 100), (127, 110), (128, 120))]
    assert list(frame[0]) == want


def test_transparent_and_outside_are_no_ops():
    for fmt in ALL_FORMATS:
        planes = random_frame(fmt, 33, 17, 5)
        before = copy_planes(planes)
        ov = random_overlay(8, 8, 1)
        ov[:, :, 3] = 0
        oracle_blend(fmt, 33, 17, planes, [dict(pixels=ov, x=3, y=3),
                                          dict(pixels=random_overlay(8, 8, 2), x=33, y=0),
                                          dict(pixels=random_overlay(8, 8, 2), x=-8, y=5),
                                          dict(pixels=random_overlay(8, 8, 2), x=0, y=17),
                                          dict(pixels=random_overlay(8, 8, 2), x=2, y=-8)])
        for p, q in zip(planes, before):
            assert np.array_equal(p, q), fmt


CASES = [
    # w, h, [(rw, rh, x, y, global_alpha, premultiplied)], opaque dest, premultiplied dest
    (64, 48, [(32, 16, 8, 8, 1.0, True)], True, False),
    (63, 47, [(31, 15, 7, 9, 1.0, True)], True, False),                 # odd everything
    (64, 48, [(40, 30, -10, -7, 1.0, True)], True, False),              # clipped left/top
    (64, 48, [(40, 30, 40, 30, 1.0, True)], True, False),               # clipped right/bottom
    (33, 21, [(80, 60, -20, -20, 1.0, True)], True, False),             # covers the whole frame
    (64, 48, [(1, 1, 5, 5, 1.0, True), (1, 1, 6, 6, 1.0, True)], True, False),
    (64, 48, [(32, 16, 8, 8, 1.0, True), (32, 16, 20, 12, 1.0, True)], True, False),   # overlap
    (64, 48, [(32, 16, 8, 8, 0.5, True), (20, 20, 30, 20, 0.8, False)], True, False),  # global alpha
    (64, 48, [(32, 16, 8, 8, 1.0, False)], True, False),                # straight source
    (64, 48, [(32, 16, 9, 7, 1.0, True)], False, False),                # non-opaque dest alpha
    (64, 48, [(32, 16, 9, 7, 0.7, True), (16, 16, 12, 10, 1.0, False)], False, True),  # premult dest
]


@pytest.mark.parametrize("fmt", ALL_FORMATS)
@pytest.mark.parametrize("case", range(len(CASES)))
def test_oracle_matches_numpy_model(fmt, case):
    w, h, rects, opaque, dprem = CASES[case]
    planes = random_frame(fmt, w, h, 100 + case, opaque=opaque)
    rectangles = [dict(pixels=random_overlay(rw, rh, 200 + 10 * case + i, premultiplied=pm),
                       x=x, y=y, global_alpha=ga, premultiplied=pm)
                  for i, (rw, rh, x, y, ga, pm) in enumerate(rects)]
    a = oracle_blend(fmt, w, h, copy_planes(planes), rectangles, dprem)
    b = model_blend(fmt, w, h, copy_planes(planes), rectangles, dprem)
    for i, (p, q) in enumerate(zip(a, b)):
        assert np.array_equal(p, q), (fmt, case, i, int((p != q).sum()))


def test_invalid_premultiplied_input_is_still_defined(oracle_lib):
    """colour > alpha never comes out of Cairo; the oracle (and the model) still agree on it."""
    ov = np.random.default_rng(9).integers(0, 256, size=(16, 16, 4), dtype=np.uint8)
    for fmt in ("NV12", "AYUV", "BGRA"):
        planes = random_frame(fmt, 32, 32, 4)
        rect = [dict(pixels=ov, x=4, y=4)]
        a = oracle_blend(fmt, 32, 32, copy_planes(planes), rect)
        b = model_blend(fmt, 32, 32, copy_planes(planes), rect)
        for p, q in zip(a, b):
            assert np.array_equal(p, q), fmt


def _sha(planes):
    h = hashlib.sha256()
    for p in planes:
        h.update(np.ascontiguousarray(p).tobytes())
    return h.hexdigest()


def test_golden_fixtures_match_oracle():
    """tests/golden/*.npz were written by tests/golden/gen_golden.py from this oracle and are
    frozen by hash in manifest.json (self-referential: see the module docstring)."""
    with open(os.path.join(GOLDEN, "manifest.json")) as f:
        manifest = json.load(f)
    assert manifest["parity"] == "unpinned"
    assert len(manifest["vectors"]) >= 9
    for v in manifest["vectors"]:
        z = np.load(os.path.join(GOLDEN, v["file"]))
        n = int(z["n_planes"])
        planes = [z[f"in{i}"].copy() for i in range(n)]
        rects = [dict(pixels=z[f"rect{i}"], x=int(z["pos"][i][0]), y=int(z["pos"][i][1]),
                      global_alpha=float(z["ga"][i]), premultiplied=bool(z["premul"][i]),
                      render_width=int(z["render"][i][0]) if "render" in z else 0,
                      render_height=int(z["render"][i][1]) if "render" in z else 0)
                 for i in range(int(z["n_rects"]))]
        out = oracle_blend(v["format"], int(z["width"]), int(z["height"]), planes, rects,
                           bool(z["dest_premul"]))
        want = [z[f"out{i}"] for i in range(n)]
        for p, q in zip(out, want):
            assert np.array_equal(p, q), v["file"]
        assert _sha(want) == v["sha256"], v["file"]


def test_baseline_byte_formula():
    """B per frame of BASELINE.md section 2."""
    assert wl.algorithmic_bytes(wl.CONFIGS[1]) == 3207168
    assert wl.algorithmic_bytes(wl.CONFIGS[2]) == 8315136
    assert wl.algorithmic_bytes(wl.CONFIGS[3]) == 32624640
    assert wl.algorithmic_bytes(wl.CONFIGS[4]) == 74096640
    assert wl.algorithmic_bytes(wl.CONFIGS[5]) == 7216128


def test_workloads_are_deterministic_and_valid_premultiplied():
    cfg = wl.CONFIGS[1]
    a, b = wl.overlay_for(cfg), wl.overlay_for(cfg)
    assert np.array_equal(a, b)
    assert (a[:, :, :3].max(axis=2) <= a[:, :, 3]).all()
    assert a[:576].max() == 0 and a[576:684, 128:1152, 3].max() == 255
    assert wl.splitmix64(0, 1)[0] == np.uint64(0xE220A8397B1DCDAF)   # published first output for seed 0


def test_gaussian_kernel_is_the_references_formula():
    """gst_ttml_blur_create_gaussian_kernel (gstttmlblur.c:28-67): normalised 2-D Gaussian in
    16.16 fixed point (truncated), symmetric, sums to just under 1.0."""
    import math
    from oracle import oracle
    for radius, sigma in ((1, 0.5), (2, 1.0), (5, 2.5)):
        k = oracle.gaussian_kernel(radius, sigma)
        size = 2 * radius + 1
        g = np.array([[math.exp(-(x * x + y * y) / (2 * sigma * sigma)) for y in range(-radius, radius + 1)]
                      for x in range(-radius, radius + 1)])
        want = np.floor(g / g.sum() * 65536.0).astype(np.int64)
        assert k.shape == (size, size)
        assert np.abs(k.astype(np.int64) - want).max() <= 1     # same formula up to the last ulp of exp()
        assert np.array_equal(k, k.T) and np.array_equal(k, k[::-1, ::-1])
        assert 65536 - size * size <= k.sum() <= 65536


def test_blur_known_answers():
    from oracle import oracle
    img = np.zeros((9, 9, 4), dtype=np.uint8)
    img[4, 4] = 255
    out = oracle.blur_argb32(img, 2, 1.0)
    k = oracle.gaussian_kernel(2, 1.0).astype(np.int64)
    want = np.clip((255 * k + 0x8000) >> 16, 0, 255)
    assert np.array_equal(out[2:7, 2:7, 3], want)           # impulse response == the kernel
    assert out[:2].max() == 0 and out[:, :2].max() == 0
    flat = np.full((12, 12, 4), 200, dtype=np.uint8)
    out = oracle.blur_argb32(flat, 2, 1.0)
    assert abs(int(out[6, 6, 0]) - 200) <= 1                 # interior of a flat field stays flat
    assert out[0, 0, 0] < 150                                # edges fade: outside is transparent


@pytest.mark.parametrize("seed", range(60))
def test_fuzz_oracle_vs_model(seed):
    """The line-structured oracle and the per-plane numpy model agree on random geometry."""
    r = np.random.default_rng(5000 + seed)
    fmt = ALL_FORMATS[seed % len(ALL_FORMATS)]
    w, h = int(r.integers(1, 120)), int(r.integers(1, 80))
    packed = fmt in PACKED
    opaque = bool(r.random() < 0.6) or not packed
    dprem = packed and bool(r.random() < 0.3)
    rects = []
    for i in range(int(r.integers(1, 6))):
        rw, rh = int(r.integers(1, w + 20)), int(r.integers(1, h + 20))
        pm = bool(r.random() < 0.7)
        rects.append(dict(pixels=random_overlay(rw, rh, int(r.integers(1 << 30)), premultiplied=pm),
                          x=int(r.integers(-rw, w + 5)), y=int(r.integers(-rh, h + 5)),
                          global_alpha=float(r.choice([1.0, 0.5, 0.99, 0.0])), premultiplied=pm))
    planes = random_frame(fmt, w, h, int(r.integers(1 << 30)), opaque=opaque)
    a = oracle_blend(fmt, w, h, copy_planes(planes), rects, dprem)
    b = model_blend(fmt, w, h, copy_planes(planes), rects, dprem)
    for i, (p, q) in enumerate(zip(a, b)):
        assert np.array_equal(p, q), (fmt, seed, i, int((p != q).sum()))


def test_oracle_under_asan_ubsan(tmp_path):
    """The C oracle over awkward geometry (1x1 frames, rectangles hanging over every border,
    exact-size allocations) built with -fsanitize=address,undefined: no out-of-bounds access,
    no signed overflow, no misaligned load."""
    import subprocess
    exe = str(tmp_path / "selftest")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["gcc", "-O1", "-g", "-std=c99", "-D_POSIX_C_SOURCE=200809L",
                           "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                           "-o", exe, os.path.join(root, "oracle", "selftest.c"),
                           os.path.join(root, "oracle", "ttmlblend_ref.c"), "-lpthread", "-lm"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 failure(s)" in r.stdout


def test_region_composition_known_answers():
    """pixman MUL_UN8 ((a*b + 0x80 + ((a*b + 0x80) >> 8)) >> 8) and Cairo's colour conversion,
    hand-computed."""
    from oracle import oracle
    regions = [dict(x=0, y=0, w=2, h=1, background_color=0xFFFFFFFF, opacity=1.0),     # opaque white
               dict(x=1, y=0, w=2, h=1, background_color=0x336699CC, opacity=1.0)]
    ov = oracle.compose_regions(regions, 4, 1)
    assert list(ov[0, 0]) == [255, 255, 255, 255]
    # 0x336699CC: a = 0xCC = 204; premultiplied shorts r = 0x33*204*257/255 + .5 -> >> 8
    a = 204
    want = [int((c / 255.0) * (a / 255.0) * 65535.0 + 0.5) >> 8 for c in (0x99, 0x66, 0x33)] + [a]
    assert list(ov[0, 2]) == want                                    # on the cleared canvas: src itself
    mul = lambda x, y: (((x * y + 0x80) >> 8) + (x * y + 0x80)) >> 8
    over_white = [min(255, s + mul(255, 255 - a)) for s in want]
    assert list(ov[0, 1]) == over_white
    assert ov[0, 3].max() == 0
    # opacity goes through a group: IN with (opacity * 65535 + 0.5) >> 8
    ov = oracle.compose_regions([dict(x=0, y=0, w=1, h=1, background_color=0xFF0000FF, opacity=0.25)], 1, 1)
    m8 = int(0.25 * 65535.0 + 0.5) >> 8
    assert list(ov[0, 0]) == [0, 0, mul(255, m8), mul(255, m8)]


# ---------------------------------------------------------------------------------------------
# rectangle scaling (gst_video_blend_scale_linear_RGBA, docs/BLENDSPEC.md section 10)

def test_scale_known_answers():
    """Hand-computed from the two ORC formulas. 2x2 -> 3x3: both increments are
    (1 << 16)/2 - 1 = 32767, so the positions are 0, 32767 (fraction 127), 65534 (still pixel
    0, fraction 255): the last source pixel is never reached exactly (254, not 255)."""
    from helpers import model_scale
    img = np.zeros((2, 2, 4), np.uint8)
    img[:, 1] = 255                                   # left column 0, right column 255
    out = oracle.scale_linear_rgba(img, 3, 3)
    assert out[..., 0].tolist() == [[0, (255 * 127) >> 8, (255 * 255) >> 8]] * 3 == [[0, 126, 254]] * 3
    img = np.zeros((2, 2, 4), np.uint8)
    img[1] = 255                                      # top row 0, bottom row 255
    out = oracle.scale_linear_rgba(img, 3, 3)
    col = [0, (255 * 127 + 128) >> 8, (255 * 255 + 128) >> 8]
    assert col == [0, 127, 254] and out[:, :, 2].T.tolist() == [col] * 3
    # a constant image stays constant, whatever the size
    img = np.full((5, 7, 4), 93, np.uint8)
    assert (oracle.scale_linear_rgba(img, 40, 3) == 93).all() and (model_scale(img, 40, 3) == 93).all()
    # one destination row / column: increments 0 -> first source row / column
    img = np.arange(3 * 4 * 4, dtype=np.uint8).reshape(3, 4, 4)
    assert np.array_equal(oracle.scale_linear_rgba(img, 1, 1)[0, 0], img[0, 0])


@pytest.mark.parametrize("seed", range(30))
def test_scale_oracle_equals_numpy_model(seed):
    from helpers import model_scale
    r = np.random.default_rng(4000 + seed)
    sw, sh = (int(v) for v in r.integers(2, 90, 2))
    dw, dh = (int(v) for v in r.integers(1, 260, 2))
    img = r.integers(0, 256, (sh, sw, 4), dtype=np.uint8)
    assert np.array_equal(oracle.scale_linear_rgba(img, dw, dh), model_scale(img, dw, dh)), (sw, sh, dw, dh)


def test_scale_line_cache_quirk_sizes():
    """Tall sources scaled down: destination rows whose 16.16 position has a zero fraction copy
    whatever the two-line cache holds (not row j). Oracle (literal loop) == model (simulation)."""
    from helpers import model_scale
    r = np.random.default_rng(7)
    for sh, dh in ((4377, 3340), (4324, 1397)):
        img = r.integers(0, 256, (sh, 3, 4), dtype=np.uint8)
        assert np.array_equal(oracle.scale_linear_rgba(img, 5, dh), model_scale(img, 5, dh))


@pytest.mark.parametrize("fmt", ("I420", "NV12", "AYUV", "BGRA", "YUY2"))
def test_scaled_rectangles_in_a_composition(fmt):
    w, h = 160, 90
    rects = [dict(pixels=random_overlay(50, 20, 31), x=10, y=50, render_width=120, render_height=33),
             dict(pixels=random_overlay(90, 60, 32, premultiplied=False), x=-7, y=-5, premultiplied=False,
                  global_alpha=0.6, render_width=40, render_height=25),
             dict(pixels=random_overlay(30, 30, 33), x=140, y=70, render_width=61, render_height=30)]
    planes = random_frame(fmt, w, h, 77)
    want = model_blend(fmt, w, h, copy_planes(planes), rects)
    got = oracle_blend(fmt, w, h, copy_planes(planes), rects)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    # scaling first and blending the result at pixel size is the same thing
    pre = [dict(r, pixels=oracle.scale_linear_rgba(r["pixels"], r["render_width"], r["render_height"]),
                render_width=0, render_height=0) for r in rects]
    again = oracle_blend(fmt, w, h, copy_planes(planes), pre)
    for a, b in zip(got, again):
        assert np.array_equal(a, b)
    assert any(not np.array_equal(a, b) for a, b in zip(got, planes))


# ---------------------------------------------------------------------------------------------
# oracle/_ref: the reference's own gstttmlblur.c, compiled from the reference tree. That tree is
# not part of this repository, so these tests run only where it has been built and skip elsewhere.

KERNEL_CASES = [(0, 0.7), (1, 0.5), (2, 1.0), (3, 1.5), (5, 2.5), (8, 4.0), (12, 3.3), (20, 10.0), (32, 8.0)]
BLUR_CASES = [(1, 1, 0.8), (2, 2, 1.0), (3, 4, 2.0), (4, 7, 3.0)]

needs_ref = pytest.mark.skipif(oracle.load_ref() is None,
                               reason="oracle/_ref not built: needs the reference's plugins/ttml/gstttmlblur.c "
                                      "(make -C oracle ref REFERENCE=<reference tree>)")


@needs_ref
@pytest.mark.parametrize("radius,sigma", KERNEL_CASES)
def test_gaussian_kernel_equals_the_references_own_code(radius, sigma):
    """The taps the reference's gst_ttml_blur_create_gaussian_kernel hands to pixman
    (gstttmlblur.c:28-67, executed) against the oracle's restatement: bit for bit, every tap,
    plus the two size parameters."""
    img = np.zeros((3, 3, 4), np.uint8)
    _, params = oracle.ref_blur_argb32(img, radius, sigma)
    size = 2 * radius + 1
    assert params[0] == params[1] == size << 16
    want = oracle.gaussian_kernel(radius, sigma).astype(np.int64).ravel()
    assert np.array_equal(params[2:], want)


@needs_ref
@pytest.mark.parametrize("seed,radius,sigma", BLUR_CASES)
def test_blur_through_the_references_call_sequence(seed, radius, sigma):
    """gst_ttml_blur_image_surface as the reference wrote it (surface -> pixman image, filter,
    PIXMAN_OP_SRC onto a cleared image of the same stride, new surface) with the convolution
    itself restated (oracle/refstub/README.md): equals tbref_blur_argb32."""
    r = np.random.default_rng(seed)
    a = r.integers(0, 256, (37, 53, 1), dtype=np.uint8)
    img = np.concatenate([(r.integers(0, 256, (37, 53, 3)) * a // 255).astype(np.uint8), a], axis=2)
    got, _ = oracle.ref_blur_argb32(img, radius, sigma)
    assert np.array_equal(got, oracle.blur_argb32(img, radius, sigma))


# ---------------------------------------------------------------------------------------------
# golden/blur_oracle.npz: the ORACLE's taps and blurred images for the cases above, frozen by hash.
# Not the reference's values (those need oracle/_ref, above); what is checked here is that the
# oracle does not drift, and that the frozen values agree with independent numpy restatements of
# the documented formulas (the Gaussian of gstttmlblur.c, pixman's convolution filter).

BLUR_ORACLE = np.load(os.path.join(GOLDEN, "blur_oracle.npz"))
BLUR_ORACLE_SHA256 = "ff08a88542170433b70a9b2b6cf0f72d07d4e9e16f492f57d47fa2113522e00a"


def _blur_oracle_sha():
    h = hashlib.sha256()
    for k in sorted(BLUR_ORACLE.files):
        h.update(k.encode())
        h.update(np.ascontiguousarray(BLUR_ORACLE[k]).tobytes())
    return h.hexdigest()


def _blur_oracle_case(key, case):
    cases = [tuple(c) for c in BLUR_ORACLE[key].tolist()]
    assert case in cases, (key, case)
    return cases.index(case)


def _numpy_convolve(img, taps):
    """pixman's convolution filter restated: window [x-r, x+r] x [y-r, y+r], outside the image
    transparent (REPEAT_NONE), 16.16 taps, (sum + 0x8000) >> 16, clipped to 0..255."""
    size = taps.shape[0]
    r = (size - 1) // 2
    h, w = img.shape[:2]
    pad = np.zeros((h + 2 * r, w + 2 * r, 4), np.int64)
    pad[r:r + h, r:r + w] = img
    tot = np.zeros((h, w, 4), np.int64)
    for i in range(size):
        for j in range(size):
            tot += int(taps[i, j]) * pad[i:i + h, j:j + w]
    return np.clip((tot + 0x8000) >> 16, 0, 255).astype(np.uint8)


def test_blur_oracle_vectors_are_frozen():
    assert str(BLUR_ORACLE["source"]).startswith("oracle/ttmlblend_ref.c")
    assert _blur_oracle_sha() == BLUR_ORACLE_SHA256


@pytest.mark.parametrize("radius,sigma", KERNEL_CASES)
def test_gaussian_kernel_matches_frozen_oracle_taps(radius, sigma):
    """tbref_gaussian_kernel equals its frozen taps bit for bit; the frozen taps are the
    normalised 2-D Gaussian in truncated 16.16 computed with numpy (up to the last ulp of exp())."""
    import math
    want = BLUR_ORACLE[f"taps{_blur_oracle_case('kernel_cases', (radius, sigma))}"].astype(np.int64)
    size = 2 * radius + 1
    assert want.shape == (size * size,)
    assert np.array_equal(oracle.gaussian_kernel(radius, sigma).astype(np.int64).ravel(), want)
    g = np.array([[math.exp(-(x * x + y * y) / (2 * sigma * sigma)) for y in range(-radius, radius + 1)]
                  for x in range(-radius, radius + 1)])
    assert np.abs(np.floor(g / g.sum() * 65536.0).astype(np.int64).ravel() - want).max() <= 1


@pytest.mark.parametrize("seed,radius,sigma", BLUR_CASES)
def test_blur_matches_frozen_oracle_images(seed, radius, sigma):
    """tbref_blur_argb32 equals its frozen output bit for bit; the frozen output is the frozen
    input convolved with the frozen taps by the numpy restatement of pixman's filter."""
    k = _blur_oracle_case("blur_cases", (seed, radius, sigma))
    img, taps, want = BLUR_ORACLE[f"blur_in{k}"], BLUR_ORACLE[f"blur_taps{k}"], BLUR_ORACLE[f"blur_out{k}"]
    size = 2 * radius + 1
    assert img.shape == want.shape == (37, 53, 4) and taps.shape == (size * size,)
    assert np.array_equal(oracle.blur_argb32(img, radius, sigma), want)
    assert np.array_equal(oracle.gaussian_kernel(radius, sigma).ravel(), taps)
    assert np.array_equal(_numpy_convolve(img, taps.reshape(size, size)), want)


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_scaled_compositions_oracle_vs_model(seed):
    """Random compositions in which some rectangles carry a render size, every format in turn:
    the line-structured oracle (scale, then gst_video_blend) against the numpy model."""
    r = np.random.default_rng(12000 + seed)
    fmt = ALL_FORMATS[seed % len(ALL_FORMATS)]
    w, h = int(r.integers(8, 200)), int(r.integers(8, 120))
    rects = []
    for i in range(int(r.integers(1, 5))):
        sw, sh = int(r.integers(2, 80)), int(r.integers(2, 60))
        pm = bool(r.integers(0, 2))
        d = dict(pixels=random_overlay(sw, sh, 50 * seed + i, premultiplied=pm), premultiplied=pm,
                 global_alpha=float(r.choice([1.0, 1.0, 0.4])))
        rw, rh = sw, sh
        if r.random() < 0.7:
            rw, rh = int(r.integers(1, 2 * w)), int(r.integers(1, 2 * h))
            d.update(render_width=rw, render_height=rh)
        d.update(x=int(r.integers(-rw, w)), y=int(r.integers(-rh, h)))
        rects.append(d)
    planes = random_frame(fmt, w, h, seed, opaque=fmt not in PACKED or bool(r.integers(0, 2)))
    want = model_blend(fmt, w, h, copy_planes(planes), rects)
    got = oracle_blend(fmt, w, h, copy_planes(planes), rects)
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), (fmt, seed, i, int((a != b).sum()))
