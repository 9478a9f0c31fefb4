"""CPU tests of the host runtime's pure logic (no GPU): the job builder (bands, windows,
classes, chunk counts, magic division, grouping), the region-box decomposition and the
row-run crop, through libfluc_ttmlblend_testhooks.so (csrc/test_hooks.cu). The properties
checked are the ones the kernels rely on: windows tile each plane exactly once, a JC_ONE
window lies inside its rectangle, a JC_COPY window touches none, the umulhi division is
exact for every item, and the byte count is BASELINE.md's formula."""
import ctypes as C
import os
import random

import numpy as np
import pytest

import __graft_entry__ as graft

HOOKS = os.path.join(graft.PKG_DIR, "csrc", "libfluc_ttmlblend_testhooks.so")

JC_COPY, JC_ONE, JC_GENERAL, JC_ONE_BULK = 0, 1, 2, 3
JF_VECTOR, JF_INPLACE, JF_DST_PREMUL, JF_FAST = 1, 2, 4, 8
ITEMS_PER_CHUNK = 1024
FMT = {"I420": 0, "NV12": 1, "AYUV": 2, "RGBA": 3, "BGRA": 4, "ARGB": 7, "Y42B": 13, "Y444": 14, "YUY2": 15,
       "GRAY8": 17, "NV16": 18, "NV24": 19, "v308": 23, "RGB": 25}


class HookRect(C.Structure):
    _fields_ = [("v0", C.c_int32), ("v1", C.c_int32), ("y0", C.c_int32), ("y1", C.c_int32)]


class HookJob(C.Structure):
    _fields_ = [("plane", C.c_int32), ("cls", C.c_int32), ("flags", C.c_int32),
                ("win_v0", C.c_int32), ("win_nv", C.c_int32), ("win_y0", C.c_int32),
                ("win_rows", C.c_int32), ("n_chunks", C.c_uint32), ("div_magic", C.c_uint32),
                ("rect_mask", C.c_uint64), ("one_rect", C.c_int32), ("grouped", C.c_int32)]


class Rect(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32)]


def load_hooks():
    if not os.path.exists(HOOKS):
        graft.build()
    lib = C.CDLL(HOOKS)
    lib.tb_hook_build_jobs.restype = C.c_int
    lib.tb_hook_build_jobs.argtypes = [C.c_int] * 5 + [C.POINTER(HookRect), C.c_int] * 3 + [
        C.POINTER(HookJob), C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
    lib.tb_hook_disjoint_cover.restype = C.c_int
    lib.tb_hook_disjoint_cover.argtypes = [C.POINTER(Rect), C.c_int, C.POINTER(Rect), C.c_int]
    lib.tb_hook_crop_runs.restype = C.c_int
    lib.tb_hook_crop_runs.argtypes = [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int,
                                      C.c_int, C.POINTER(Rect), C.c_int]
    lib.tb_hook_pack_layouts.restype = C.c_int
    lib.tb_hook_pack_layouts.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_int,
                                         C.POINTER(HookRect), C.POINTER(C.c_int32), C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.tb_hook_scale_row_plan.restype = C.c_int
    lib.tb_hook_scale_row_plan.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int32)]
    lib.tb_hook_interval_set.restype = C.c_int
    lib.tb_hook_interval_set.argtypes = [C.POINTER(C.c_uint64), C.c_int, C.POINTER(C.c_int32),
                                         C.POINTER(C.c_uint64), C.c_int]
    return lib


@pytest.fixture(scope="module")
def hooks():
    return load_hooks()


def plane_geometry(fmt, W, H):
    """[(row_bytes, rows)] per plane -- restated from the format table in docs/BLENDSPEC.md."""
    cw, ch = (W + 1) // 2, (H + 1) // 2
    return {
        "I420": [(W, H), (cw, ch), (cw, ch)],
        "NV12": [(W, H), (2 * cw, ch)],
        "Y42B": [(W, H), (cw, H), (cw, H)],
        "Y444": [(W, H)] * 3,
        "NV16": [(W, H), (2 * cw, H)],
        "NV24": [(W, H), (2 * W, H)],
        "YUY2": [(4 * cw, H)],
        "GRAY8": [(W, H)],
        "AYUV": [(4 * W, H)], "RGBA": [(4 * W, H)], "BGRA": [(4 * W, H)], "ARGB": [(4 * W, H)],
        "RGB": [(3 * W, H)], "v308": [(3 * W, H)],
    }[fmt]


def plane_rects(fmt, W, H, rects):
    """Per plane, the (v0, v1, y0, y1) span the prepare gives each pixel rectangle (x, y, w, h) of
    the composition form, clipped to the frame: its byte columns widened to whole vectors, and for
    the chroma planes the samples it sites (restated from prepare_rect / prepare_chroma)."""
    bpp = {"AYUV": 4, "RGBA": 4, "BGRA": 4, "ARGB": 4, "RGB": 3, "v308": 3}
    sub = {"I420": (2, 2), "NV12": (2, 2), "Y444": (1, 1)}
    out = [[] for _ in plane_geometry(fmt, W, H)]
    cdiv = lambda a, b: -(-a // b)
    for (x, y, w, h) in rects:
        x0, y0, x1, y1 = max(x, 0), max(y, 0), min(x + w, W), min(y + h, H)
        b = bpp.get(fmt, 1)
        out[0].append((b * x0 // 16, cdiv(b * x1, 16), y0, y1))
        if fmt in sub:
            sx, sy = sub[fmt]
            bx0, bx1, by0, by1 = cdiv(x0, sx), cdiv(x1, sx), cdiv(y0, sy), cdiv(y1, sy)
            e = 2 if fmt == "NV12" else 1
            for pl in range(1, len(out)):
                out[pl].append((e * bx0 // 16, cdiv(e * bx1, 16), by0, by1))
    return out


def build(hooks, fmt, W, H, rects_per_plane, windowed=False, misalign=False):
    arrs, ns = [], []
    for pl in range(3):
        rr = rects_per_plane[pl] if pl < len(rects_per_plane) else []
        a = (HookRect * max(1, len(rr)))(*[HookRect(*r) for r in rr])
        arrs.append(a)
        ns.append(len(rr))
    out = (HookJob * 4096)()
    algo = C.c_uint64(0)
    cpf = C.c_uint32(0)
    n = hooks.tb_hook_build_jobs(FMT[fmt], W, H, int(windowed), int(misalign),
                                 arrs[0], ns[0], arrs[1], ns[1], arrs[2], ns[2],
                                 out, 4096, C.byref(algo), C.byref(cpf))
    assert n >= 0
    return [out[i] for i in range(n)], algo.value, cpf.value


def check_tiling(fmt, W, H, rects_per_plane, jobs, windowed):
    """Every vector of every plane row is in exactly one window (out of place), or exactly the
    vectors under a rectangle are (windowed); classes agree with the rectangles."""
    geo = plane_geometry(fmt, W, H)
    for pl, (row_bytes, rows) in enumerate(geo):
        nv_row = (row_bytes + 15) // 16
        cover = np.zeros((rows, nv_row), np.int32)
        under = np.zeros((rows, nv_row), np.int32)
        rr = rects_per_plane[pl] if pl < len(rects_per_plane) else []
        for (v0, v1, y0, y1) in rr:
            under[max(0, y0):max(0, min(rows, y1)), max(0, v0):max(0, min(nv_row, v1))] += 1
        for j in jobs:
            if j.plane != pl:
                continue
            assert 0 <= j.win_v0 and j.win_v0 + j.win_nv <= nv_row and j.win_nv > 0
            assert 0 <= j.win_y0 and j.win_y0 + j.win_rows <= rows and j.win_rows > 0
            sl = (slice(j.win_y0, j.win_y0 + j.win_rows), slice(j.win_v0, j.win_v0 + j.win_nv))
            cover[sl] += 1
            items = j.win_nv * j.win_rows
            assert j.n_chunks == (items + ITEMS_PER_CHUNK - 1) // ITEMS_PER_CHUNK
            if j.cls == JC_COPY:
                assert (under[sl] == 0).all() and j.rect_mask == 0
            elif j.cls in (JC_ONE, JC_ONE_BULK):
                v0, v1, y0, y1 = rr[j.one_rect]
                assert j.rect_mask == 1 << j.one_rect
                assert v0 <= j.win_v0 and j.win_v0 + j.win_nv <= v1      # no per-vector tests needed
                assert y0 <= j.win_y0 and j.win_y0 + j.win_rows <= y1
                assert (under[sl] == 1).all()
                if j.cls == JC_ONE_BULK:
                    assert row_bytes % 16 == 0      # the table kernel treats it as JC_ONE
            else:
                assert j.cls == JC_GENERAL
                # the mask names the whole column cluster (a window split off at the ragged last
                # vector keeps it): a superset of the rectangles over the window, all of them
                # spanning the band's rows; the kernel tests columns per vector
                need = rows_ok = 0
                for i, (v0, v1, y0, y1) in enumerate(rr):
                    spans = y0 <= j.win_y0 and y1 >= j.win_y0 + j.win_rows
                    if spans:
                        rows_ok |= 1 << i
                    if spans and v0 < j.win_v0 + j.win_nv and v1 > j.win_v0:
                        need |= 1 << i
                assert j.rect_mask & need == need and j.rect_mask & ~rows_ok == 0
                assert bin(j.rect_mask).count("1") >= 2
            # ragged last vector column never goes to the whole-vector kernel
            if j.flags & JF_FAST:
                assert (j.win_v0 + j.win_nv) * 16 <= row_bytes and (j.flags & JF_VECTOR)
            assert bool(j.flags & JF_INPLACE) == windowed
            # umulhi(item, magic) == item // nv for every item the kernel can see
            if j.win_nv > 1:
                padded = j.n_chunks * ITEMS_PER_CHUNK
                probe = np.unique(np.concatenate([
                    np.arange(0, min(padded, 4096)), np.arange(max(0, padded - 4096), padded),
                    np.arange(0, padded, max(1, padded // 2048))])).astype(np.uint64)
                assert ((probe * np.uint64(j.div_magic)) >> np.uint64(32) == probe // np.uint64(j.win_nv)).all()
            else:
                assert j.div_magic == 0
        if windowed:
            assert ((cover == 1) == (under > 0)).all() and cover.max(initial=0) <= 1
        else:
            assert (cover == 1).all()


def test_no_overlay_is_one_copy_window_per_plane(hooks):
    jobs, algo, cpf = build(hooks, "NV12", 3840, 2160, [[], []])
    assert [(j.plane, j.cls, j.win_nv, j.win_rows) for j in jobs] == [(0, JC_COPY, 240, 2160), (1, JC_COPY, 240, 1080)]
    assert algo == 2 * 3840 * 2160 * 3 // 2
    assert cpf == sum(j.n_chunks for j in jobs) == 507 + 254
    check_tiling("NV12", 3840, 2160, [[], []], jobs, False)


def test_config3_bands_are_bulk_and_grouped(hooks):
    # full-width regions of BASELINE config 3 on the Y and UV planes
    y = [(0, 240, 1728, 2088), (0, 240, 72, 216)]
    uv = [(0, 240, 864, 1044), (0, 240, 36, 108)]
    jobs, algo, cpf = build(hooks, "NV12", 3840, 2160, [y, uv])
    cls = [(j.plane, j.win_y0, j.cls) for j in jobs]
    assert cls == [(0, 0, JC_COPY), (0, 72, JC_ONE_BULK), (0, 216, JC_COPY), (0, 1728, JC_ONE_BULK), (0, 2088, JC_COPY),
                   (1, 0, JC_COPY), (1, 36, JC_ONE_BULK), (1, 108, JC_COPY), (1, 864, JC_ONE_BULK), (1, 1044, JC_COPY)]
    assert all(j.grouped and (j.flags & JF_FAST) for j in jobs)
    assert cpf == sum(j.n_chunks for j in jobs)
    # the hook's fake Prepared has overlay_px == 0, so only the frame part is counted
    assert algo == 2 * 12441600
    check_tiling("NV12", 3840, 2160, [y, uv], jobs, False)


def test_narrow_region_becomes_copy_one_copy(hooks):
    y = [(12, 108, 864, 1026)]
    jobs, _, _ = build(hooks, "I420", 1920, 1080, [y, [], []])
    band = [(j.cls, j.win_v0, j.win_nv) for j in jobs if j.plane == 0 and j.win_y0 == 864]
    assert band == [(JC_COPY, 0, 12), (JC_ONE_BULK, 12, 96), (JC_COPY, 108, 12)]
    check_tiling("I420", 1920, 1080, [y, [], []], jobs, False)
    # in place: only the window under the rectangle exists
    jobs, algo, _ = build(hooks, "I420", 1920, 1080, [y, [], []], windowed=True)
    assert [(j.plane, j.cls, j.win_v0, j.win_nv, j.win_y0, j.win_rows) for j in jobs] == [(0, JC_ONE_BULK, 12, 96, 864, 162)]
    assert algo == 2 * 96 * 16 * 162
    check_tiling("I420", 1920, 1080, [y, [], []], jobs, True)


def test_rectangles_sharing_columns_form_a_general_window(hooks):
    y = [(10, 60, 100, 300), (40, 90, 200, 400), (100, 110, 150, 250)]
    jobs, _, _ = build(hooks, "GRAY8", 1920, 1080, [y])
    mid = [(j.cls, j.win_v0, j.win_nv, j.rect_mask) for j in jobs if j.win_y0 == 200]
    assert mid == [(JC_COPY, 0, 10, 0), (JC_GENERAL, 10, 80, 0b011), (JC_COPY, 90, 10, 0),
                   (JC_ONE_BULK, 100, 10, 0b100), (JC_COPY, 110, 10, 0)]
    check_tiling("GRAY8", 1920, 1080, [y], jobs, False)


def test_ragged_last_vector_goes_to_the_byte_kernel(hooks):
    # 1279 px wide luma: 79 whole vectors + a 15-byte tail column
    y = [(0, 80, 600, 700)]
    jobs, algo, cpf = build(hooks, "I420", 1279, 719, [y, [], []])
    tails = [j for j in jobs if j.plane == 0 and j.win_v0 == 79]
    assert tails and all(j.win_nv == 1 and not (j.flags & JF_FAST) and (j.flags & JF_VECTOR) and not j.grouped
                         for j in tails)
    assert all(j.cls != JC_ONE_BULK for j in jobs if j.plane == 0)
    assert algo == 2 * (1279 * 719 + 2 * 640 * 360)
    check_tiling("I420", 1279, 719, [y, [], []], jobs, False)


def test_misaligned_frames_never_take_the_vector_path(hooks):
    y = [(0, 120, 100, 200)]
    jobs, _, cpf = build(hooks, "GRAY8", 1920, 1080, [y], misalign=True)
    assert cpf == 0 and all(not (j.flags & (JF_FAST | JF_VECTOR)) and not j.grouped for j in jobs)
    check_tiling("GRAY8", 1920, 1080, [y], jobs, False)


def test_too_many_bands_fall_back_to_the_table_kernel(hooks):
    y = [(0, 120, 10 * i, 10 * i + 5) for i in range(40)]       # 80 bands > 64 (the first starts at row 0)
    jobs, _, cpf = build(hooks, "GRAY8", 1920, 1080, [y])
    assert len(jobs) == 80 and cpf == 0 and not any(j.grouped for j in jobs)
    check_tiling("GRAY8", 1920, 1080, [y], jobs, False)


@pytest.mark.parametrize("seed", range(24))
def test_random_layouts_tile_every_plane_once(hooks, seed):
    rnd = random.Random(seed)
    fmt = rnd.choice(sorted(FMT))
    W, H = rnd.choice([(64, 48), (333, 97), (1279, 719), (1920, 1080), (17, 5)])
    geo = plane_geometry(fmt, W, H)
    rects = []
    n = rnd.randrange(0, 7)
    for row_bytes, rows in geo:
        nv = (row_bytes + 15) // 16
        rr = []
        for _ in range(n):
            v0 = rnd.randrange(-2, nv)
            y0 = rnd.randrange(-3, rows)
            rr.append((v0, v0 + rnd.randrange(1, nv + 3), y0, y0 + rnd.randrange(1, rows + 3)))
        rects.append(rr)
    for windowed in (False, True):
        jobs, algo, _ = build(hooks, fmt, W, H, rects, windowed=windowed)
        check_tiling(fmt, W, H, rects, jobs, windowed)
        if not windowed:
            assert algo == 2 * sum(rb * r for rb, r in geo)


def pieces(jobs, plane=0):
    return [(j.win_v0, j.win_nv, j.win_y0, j.win_rows, j.cls, j.grouped) for j in jobs if j.plane == plane]


# Frames above 4K (tests/test_gpu_geometry.py). push_window cuts a window into pieces of at most
# max_rows rows so that umulhi (item, magic) stays exact, and make_groupable sends a layout to the
# table kernel when a full group of frames would not divide exactly. These pin which pieces and
# which kernel the GPU cases reach: a change to either function shows here first.

def test_8k_packed_windows_are_cut_into_1344_row_pieces(hooks):
    rects = [(0, 200, 7680, 1500), (2000, 1600, 1200, 600)]
    for fmt in ("RGBA", "BGRA", "AYUV", "ARGB"):
        rr = plane_rects(fmt, 7680, 4320, rects)
        jobs, _, cpf = build(hooks, fmt, 7680, 4320, rr, windowed=True)
        assert pieces(jobs) == [(0, 1920, 200, 1344, JC_ONE_BULK, 1), (0, 1920, 1544, 56, JC_ONE_BULK, 1),
                                (0, 1920, 1600, 100, JC_GENERAL, 1), (500, 300, 1700, 500, JC_ONE_BULK, 1)]
        jobs, _, cpf = build(hooks, fmt, 7680, 4320, rr)
        assert cpf > 0 and all(j.grouped for j in jobs)
        assert [(j.win_y0, j.win_rows) for j in jobs if j.win_nv == 1920] == [
            (0, 200), (200, 1344), (1544, 56), (1600, 100), (2200, 1344), (3544, 776)]
    check_tiling("BGRA", 7680, 4320, rr, jobs, False)
    # the same frame with the tall rectangle moved by (3, 37): the pieces start elsewhere
    moved = plane_rects("BGRA", 7680, 4320, [(3, 237, 7680, 1500), (2000, 1600, 1200, 600)])
    jobs, _, _ = build(hooks, "BGRA", 7680, 4320, moved, windowed=True)
    assert pieces(jobs)[:2] == [(0, 1920, 237, 1344, JC_ONE_BULK, 1), (0, 1920, 1581, 19, JC_ONE_BULK, 1)]
    check_tiling("BGRA", 7680, 4320, moved, jobs, True)


def test_8k_three_byte_windows_are_cut_into_2519_row_pieces(hooks):
    rects = [(0, 200, 7680, 2700), (2000, 2800, 1200, 600)]
    for fmt in ("RGB", "v308"):
        rr = plane_rects(fmt, 7680, 4320, rects)
        jobs, _, _ = build(hooks, fmt, 7680, 4320, rr, windowed=True)
        assert pieces(jobs) == [(0, 1440, 200, 2519, JC_ONE_BULK, 1), (0, 1440, 2719, 81, JC_ONE_BULK, 1),
                                (0, 1440, 2800, 100, JC_GENERAL, 1), (375, 225, 2900, 500, JC_ONE_BULK, 1)]
        # out of place the chunk count makes a full group inexact: the table kernel
        jobs, _, cpf = build(hooks, fmt, 7680, 4320, rr)
        assert cpf == 0 and not any(j.grouped for j in jobs) and all(j.flags & JF_FAST for j in jobs)
        assert [(j.win_y0, j.win_rows) for j in jobs if j.win_nv == 1440][:3] == [(0, 200), (200, 2519), (2719, 81)]
    check_tiling("RGB", 7680, 4320, rr, jobs, False)


def test_8k_planar_windows_are_not_cut(hooks):
    rects = [(0, 200, 7680, 1500), (2000, 1600, 1200, 600)]
    for fmt in ("NV12", "I420"):
        rr = plane_rects(fmt, 7680, 4320, rects)
        for windowed in (False, True):
            jobs, _, cpf = build(hooks, fmt, 7680, 4320, rr, windowed=windowed)
            assert cpf > 0 and all(j.grouped for j in jobs)
            assert (0, 480, 200, 1400, JC_ONE_BULK, 1) in pieces(jobs)
            assert all(j.win_rows < 2500 or j.cls == JC_COPY for j in jobs)


def test_8k_rectangle_over_the_right_and_bottom_edges(hooks):
    rr = plane_rects("BGRA", 7680, 4320, [(300, 2820, 7600, 1600)])
    jobs, _, cpf = build(hooks, "BGRA", 7680, 4320, rr)
    assert cpf == 0 and pieces(jobs) == [(0, 1920, 0, 1344, JC_COPY, 0), (0, 1920, 1344, 1344, JC_COPY, 0),
                                         (0, 1920, 2688, 132, JC_COPY, 0), (0, 75, 2820, 1500, JC_COPY, 0),
                                         (75, 1845, 2820, 1500, JC_ONE_BULK, 0)]
    jobs, _, cpf = build(hooks, "BGRA", 7680, 4320, rr, windowed=True)
    assert cpf > 0 and pieces(jobs) == [(75, 1845, 2820, 1500, JC_ONE_BULK, 1)]


@pytest.mark.parametrize("fmt,W,x,w", [("RGBA", 8192, 3000, 1500), ("Y444", 8192, 3000, 1500), ("RGB", 7680, 0, 4096)])
def test_8k_geometries_that_fall_back_to_the_table_kernel(hooks, fmt, W, x, w):
    rr = plane_rects(fmt, W, 4320, [(x, 1080, w, 2160)])
    jobs, _, cpf = build(hooks, fmt, W, 4320, rr)
    assert cpf == 0 and not any(j.grouped for j in jobs) and all(j.flags & JF_FAST for j in jobs)
    jobs, _, cpf = build(hooks, fmt, W, 4320, rr, windowed=True)
    assert cpf > 0 and all(j.grouped for j in jobs)              # in place they stay grouped


def test_near_the_width_limit(hooks):
    # 32764 BGRA: 8191 vectors a row, 64-row pieces; 13 under rows 102-921. Out of place group bands,
    # in place (fewer chunks a frame) the table kernel
    rr = plane_rects("BGRA", 32764, 1024, [(0, 102, 32764, 819)])
    jobs, _, cpf = build(hooks, "BGRA", 32764, 1024, rr)
    under = [p for p in pieces(jobs) if p[4] == JC_ONE_BULK]
    assert cpf > 0 and all(j.grouped for j in jobs) and len(under) == 13
    assert [p[2:4] for p in under] == [(102 + 64 * k, 64) for k in range(12)] + [(870, 51)]
    jobs, _, cpf = build(hooks, "BGRA", 32764, 1024, rr, windowed=True)
    assert cpf == 0 and [p[2:] for p in pieces(jobs)] == [(102 + 64 * k, 64, JC_ONE_BULK, 0) for k in range(12)] + [
        (870, 51, JC_ONE_BULK, 0)]
    # 32764 AYUV under rows 102-358: four pieces, grouped both ways
    rr = plane_rects("AYUV", 32764, 1024, [(0, 102, 32764, 256)])
    for windowed in (False, True):
        jobs, _, cpf = build(hooks, "AYUV", 32764, 1024, rr, windowed=windowed)
        assert cpf > 0 and [p[2:4] for p in pieces(jobs) if p[4] == JC_ONE_BULK] == [(102, 64), (166, 64), (230, 64), (294, 64)]
    # 32767 wide: 2047 whole vectors and a 15-byte tail column for the byte kernel
    for fmt in ("GRAY8", "I420"):
        rr = plane_rects(fmt, 32767, 512, [(0, 100, 32767, 300)])
        for windowed in (False, True):
            jobs, _, cpf = build(hooks, fmt, 32767, 512, rr, windowed=windowed)
            tail = [j for j in jobs if j.win_v0 == 2047]
            assert cpf > 0 and tail and all(j.plane == 0 and j.win_nv == 1 and not j.grouped and not (j.flags & JF_FAST)
                                            for j in tail)
            assert all(j.grouped for j in jobs if j.win_v0 != 2047)
    # 15360 RGBA: 3840 vectors a row, 312-row pieces; out of place the table kernel
    rr = plane_rects("RGBA", 15360, 8640, [(0, 2000, 15360, 1000)])
    jobs, _, cpf = build(hooks, "RGBA", 15360, 8640, rr)
    assert cpf == 0 and [p[2:4] for p in pieces(jobs) if p[4] == JC_ONE_BULK] == [(2000, 312), (2312, 312), (2624, 312), (2936, 64)]
    jobs, _, cpf = build(hooks, "RGBA", 15360, 8640, rr, windowed=True)
    assert cpf > 0 and [p[2:4] for p in pieces(jobs)] == [(2000, 312), (2312, 312), (2624, 312), (2936, 64)]
    rr = plane_rects("RGBA", 15360, 8640, [(0, 2000, 15360, 4320)])
    jobs, _, cpf = build(hooks, "RGBA", 15360, 8640, rr, windowed=True)
    assert cpf == 0 and len(jobs) == 14


@pytest.mark.parametrize("fmt,W,H,rects", [
    ("BGRA", 7680, 4320, [(0, 200, 7680, 1500), (2000, 1600, 1200, 600)]),
    ("RGB", 7680, 4320, [(0, 200, 7680, 2700), (2000, 2800, 1200, 600)]),
    ("RGBA", 15360, 8640, [(0, 2000, 15360, 1000), (5000, 1500, 3000, 3000)]),
    ("BGRA", 32764, 2048, [(0, 102, 32764, 1024), (100, 1500, 200, 300)]),
])
def test_large_frames_tile_and_divide_exactly(hooks, fmt, W, H, rects):
    """check_tiling (every window once, classes, the umulhi probe over each window's items) on the
    geometries above 4K; its cover arrays are too large at 32768 x 32768."""
    rr = plane_rects(fmt, W, H, rects)
    for windowed in (False, True):
        jobs, _, _ = build(hooks, fmt, W, H, rr, windowed=windowed)
        assert any(j.win_rows == max_rows_of(j.win_nv) for j in jobs)
        check_tiling(fmt, W, H, rr, jobs, windowed)


def max_rows_of(nv):
    magic = ((1 << 32) + nv - 1) // nv
    e = magic * nv - (1 << 32)
    return max(1, min(min(((1 << 32) - 1) // e if e else 1 << 31, 1 << 31) // nv, 1 << 30))


# ---------------------------------------------------------------------------------------------

def cover_mask(rects, W=64, H=64):
    m = np.zeros((H, W), np.int32)
    for r in rects:
        m[r.y:r.y + r.h, r.x:r.x + r.w] += 1
    return m


def disjoint(hooks, rects):
    a = (Rect * len(rects))(*[Rect(*r) for r in rects])
    out = (Rect * 1024)()
    n = hooks.tb_hook_disjoint_cover(a, len(rects), out, 1024)
    assert n >= 0
    return [out[i] for i in range(n)]


def test_disjoint_cover_simple_cases(hooks):
    got = disjoint(hooks, [(0, 0, 10, 10)])
    assert [(r.x, r.y, r.w, r.h) for r in got] == [(0, 0, 10, 10)]
    # two side-by-side boxes of equal rows that touch merge into one
    got = disjoint(hooks, [(0, 0, 10, 10), (10, 0, 5, 10)])
    assert [(r.x, r.y, r.w, r.h) for r in got] == [(0, 0, 15, 10)]
    # a cross becomes three disjoint rectangles
    got = disjoint(hooks, [(4, 0, 4, 12), (0, 4, 12, 4)])
    assert sorted((r.x, r.y, r.w, r.h) for r in got) == [(0, 4, 12, 4), (4, 0, 4, 4), (4, 8, 4, 4)]


@pytest.mark.parametrize("seed", range(16))
def test_disjoint_cover_covers_the_same_pixels_once(hooks, seed):
    rnd = random.Random(100 + seed)
    rects = []
    for _ in range(rnd.randrange(1, 9)):
        x, y = rnd.randrange(0, 50), rnd.randrange(0, 50)
        rects.append((x, y, rnd.randrange(1, 64 - x), rnd.randrange(1, 64 - y)))
    got = disjoint(hooks, rects)
    want = cover_mask([Rect(*r) for r in rects]) > 0
    m = cover_mask(got)
    assert m.max() == 1 and ((m == 1) == want).all()


def crop(hooks, first, last, min_gap=16, max_runs=8):
    n = len(first)
    out = (Rect * 64)()
    k = hooks.tb_hook_crop_runs((C.c_int32 * n)(*first), (C.c_int32 * n)(*last), n, min_gap, max_runs, out, 64)
    assert k >= 0
    return [(out[i].x, out[i].y, out[i].w, out[i].h) for i in range(k)]


def test_crop_runs(hooks):
    W = 100
    empty = (W, -1)
    rows = [empty] * 200
    for y in range(10, 30):
        rows[y] = (20, 59)
    rows[15] = (5, 70)
    for y in range(100, 120):
        rows[y] = (40, 41)
    first, last = zip(*rows)
    assert crop(hooks, first, last) == [(5, 10, 66, 20), (40, 100, 2, 20)]
    # gaps below min_gap are bridged, rows in between included
    rows[35] = (0, 99)
    first, last = zip(*rows)
    assert crop(hooks, first, last) == [(0, 10, 100, 26), (40, 100, 2, 20)]
    # the run limit merges the closest pair
    assert crop(hooks, first, last, max_runs=1) == [(0, 10, 100, 110)]
    # a fully transparent rectangle yields nothing
    assert crop(hooks, [W] * 50, [-1] * 50) == []


@pytest.mark.parametrize("seed", range(8))
def test_crop_runs_keeps_every_non_transparent_pixel(hooks, seed):
    rnd = random.Random(200 + seed)
    W, H = 80, 300
    first, last = [], []
    for y in range(H):
        if rnd.random() < 0.7:
            first.append(W)
            last.append(-1)
        else:
            a = rnd.randrange(0, W)
            first.append(a)
            last.append(rnd.randrange(a, W))
    runs = crop(hooks, first, last, min_gap=rnd.choice([1, 4, 16]), max_runs=rnd.choice([1, 3, 8]))
    m = np.zeros((H, W), bool)
    for (x, y, w, h) in runs:
        assert not m[y:y + h, x:x + w].any()           # disjoint
        m[y:y + h, x:x + w] = True
    for y in range(H):
        if last[y] >= first[y]:
            assert m[y, first[y]:last[y] + 1].all()
    assert runs == sorted(runs, key=lambda r: r[1])


# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("sh,dh", [(2, 3), (2, 1), (90, 29), (45, 90), (64, 33), (53, 70), (1080, 2160),
                                   (2160, 1080), (4377, 3340), (4324, 1397), (3908, 2787)])
def test_scale_row_plan_is_the_simulated_line_cache(hooks, sh, dh):
    """The runtime's row plan for gst_video_blend_scale_linear_RGBA equals the independent
    simulation in tests/helpers.py; the last three sizes contain rows where upstream's
    two-line cache holds other rows than (j, j+1)."""
    from helpers import model_scale_rows
    out = (C.c_int32 * (3 * dh))()
    assert hooks.tb_hook_scale_row_plan(sh, dh, out) == dh
    got = [tuple(out[3 * i:3 * i + 3]) for i in range(dh)]
    want = model_scale_rows(sh, dh)
    assert got == want
    assert all(0 <= a < sh and 0 <= b < sh and 0 <= p <= 255 for a, b, p in got)
    if sh >= 3000:
        y_inc = ((sh - 1) << 16) // (dh - 1) - 1
        naive = [((i * y_inc) >> 16, (i * y_inc) >> 16, 0) if (i * y_inc) & 0xffff == 0 else
                 ((i * y_inc) >> 16, ((i * y_inc) >> 16) + 1, ((i * y_inc) & 0xffff) >> 8) for i in range(dh)]
        assert naive != got          # the quirk is really exercised


@pytest.mark.parametrize("dh", [3, 1000, 32767])
def test_scale_row_plan_at_the_largest_source_height(hooks, dh):
    """32768 source rows is the most a scaled rectangle may have: (32768 - 1) << 16 and the
    plan's accumulator still fit in 32 bits, and the runtime's plan equals the model's. One
    row more overflows them, so overlay_install refuses such a rectangle (docs/BLENDSPEC.md
    section 10; tests/test_gpu_cue_kernels.py checks the refusal)."""
    from helpers import model_scale_rows
    sh = 32768
    assert ((sh - 1) << 16) < 2 ** 31 and (dh - 1) * (((sh - 1) << 16) // max(dh - 1, 1)) < 2 ** 31
    out = (C.c_int32 * (3 * dh))()
    assert hooks.tb_hook_scale_row_plan(sh, dh, out) == dh
    got = np.frombuffer(out, dtype=np.int32).reshape(dh, 3)
    want = np.array(model_scale_rows(sh, dh), dtype=np.int32)
    assert np.array_equal(got, want)
    assert got[-1, 0] >= sh - 2 and got[:, :2].max() < sh       # reaches the bottom, stays inside


# ---------------------------------------------------------------------------------------------

def pack(hooks, W, H, ov, rects, strides):
    n = len(ov)
    ids = (C.c_uint64 * n)()
    launch = (C.c_int32 * n)()
    lists = C.c_int32(0)
    k = hooks.tb_hook_pack_layouts(W, H, n, (C.c_int32 * n)(*ov), len(rects),
                                   (HookRect * len(rects))(*[HookRect(*r) for r in rects]),
                                   (C.c_int32 * n)(*strides), ids, launch, C.byref(lists))
    assert k >= 0, k
    return k, list(ids), list(launch), lists.value


def test_layouts_are_shared_and_canonical(hooks):
    W, H = 1920, 1080
    box = (12, 108, 864, 1026)
    # 6 frames: overlays 0 and 1 have the SAME rectangle, overlay 2 another one
    k, ids, launch, lists = pack(hooks, W, H, [0, 0, 1, 1, 2, 2], [box, box, (12, 100, 800, 900)],
                                 [1920] * 6)
    assert ids[0] == ids[1] == ids[2] == ids[3]          # one layout per overlay, one id per band list
    assert ids[4] == ids[5] != ids[0]
    assert k == 1 and set(launch) == {0} and lists == 2   # one launch, two band lists
    # another stride is another layout (and another launch: strides are per launch)
    k, ids, launch, lists = pack(hooks, W, H, [0, 0, 0], [box], [1920, 2048, 1920])
    assert ids[0] == ids[2] != ids[1]
    assert k == 2 and launch[0] == launch[2] != launch[1]


def test_multi_launch_limits(hooks):
    W, H = 1920, 1080
    # 100 frames of ONE layout: 64 frames per launch
    k, ids, launch, lists = pack(hooks, W, H, [0] * 100, [(12, 108, 864, 1026)], [1920] * 100)
    assert len(set(ids)) == 1 and k == 2 and lists == 2
    assert launch.count(0) == 64 and launch.count(1) == 36
    # 60 distinct layouts of 5 bands each (copy rows above, copy | one | copy, copy rows below)
    # = 300 bands: one launch; 9 bands each (two text lines of different width) would not fit 576
    rects = [(10 + i % 7, 100 + i, 800 + i, 900 + i) for i in range(60)]
    k, ids, launch, lists = pack(hooks, W, H, list(range(60)), rects, [1920] * 60)
    assert len(set(ids)) == 60 and k == 1 and lists == 60
    rects = [(10 + i % 7, 100 + i, 40 + 6 * i, 60 + 6 * i) for i in range(64)]
    k, ids, launch, lists = pack(hooks, W, H, list(range(64)) * 2, rects, [1920] * 128)
    # 128 frames, 64 layouts x 5 bands = 320 bands: frames cap (64) decides -> 2 launches,
    # and the second pass over the same overlays reuses the band lists already in a launch
    assert k == 2 and lists in (64, 128) and launch.count(0) == 64 and launch.count(1) == 64


def _interval_ops(hooks, ops):
    """ops: [(kind, lo, hi)], kind 0 add / 1 query -> (answers, ranges held at the end)"""
    flat = (C.c_uint64 * (3 * len(ops)))(*[v for op in ops for v in op])
    out = (C.c_int32 * max(1, len(ops)))()
    ranges = (C.c_uint64 * 4096)()
    n = hooks.tb_hook_interval_set(flat, len(ops), out, ranges, 2048)
    nq = sum(1 for op in ops if op[0] == 1)
    return [out[i] for i in range(nq)], [(ranges[2 * k], ranges[2 * k + 1]) for k in range(n)]


def test_interval_set_simple(hooks):
    """The range set behind the batch hazard check (frames that write / read what a queued frame
    writes must not share its launch): half-open ranges, touching ranges merge."""
    ans, held = _interval_ops(hooks, [
        (1, 0, 100),                 # empty set
        (0, 100, 200), (1, 0, 100), (1, 199, 300), (1, 200, 300), (1, 150, 160),
        (0, 300, 400), (1, 200, 300), (0, 200, 300), (1, 250, 251),
        (0, 1000, 1100), (0, 50, 60), (1, 60, 100), (1, 59, 61),
    ])
    assert ans == [0, 0, 1, 0, 1, 0, 1, 0, 1]
    assert held == [(50, 60), (100, 400), (1000, 1100)]


@pytest.mark.parametrize("seed", range(20))
def test_interval_set_against_a_bitmap(hooks, seed):
    rnd = random.Random(7000 + seed)
    size = 4000
    bitmap = np.zeros(size, dtype=bool)
    ops, want = [], []
    for _ in range(300):
        lo = rnd.randrange(0, size - 1)
        hi = min(size, lo + rnd.choice((1, 2, 5, 40, 300)))
        if rnd.random() < 0.5:
            ops.append((0, lo, hi))
            bitmap[lo:hi] = True
        else:
            ops.append((1, lo, hi))
            want.append(int(bitmap[lo:hi].any()))
    ans, held = _interval_ops(hooks, ops)
    assert ans == want
    covered = np.zeros(size, dtype=bool)
    prev_hi = -1
    for lo, hi in held:
        assert lo < hi and lo > prev_hi          # sorted, disjoint, not even touching
        covered[lo:hi] = True
        prev_hi = hi
    assert np.array_equal(covered, bitmap)
