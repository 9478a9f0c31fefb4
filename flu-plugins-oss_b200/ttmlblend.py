"""ctypes binding of libfluc_ttmlblend.so (include/fluc_ttmlblend.h).

Thin on purpose: every method is one C-ABI call. The library is the product;
this module exists so that tests/ and bench.py can drive it the way an element
written in C would (the cgo/ctypes stub a maintainer adds is in INTEGRATION.md).
There is no CPU fallback: if the shared library is missing, or no CUDA device
is usable, construction raises.

Reference interface mirrored (argument meaning / error behaviour):
  gst_video_overlay_composition_blend / gst_video_blend (gst-plugins-base), fed
  by ttmlrender's gen_buffer output, /root/reference/plugins/ttml/gstttmlrender.c:1427-1478.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Iterable, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libfluc_ttmlblend.so")

FORMATS = {
    "I420": 0, "NV12": 1, "AYUV": 2, "RGBA": 3, "BGRA": 4,
    "YV12": 5, "NV21": 6, "ARGB": 7, "ABGR": 8,
    "RGBx": 9, "BGRx": 10, "xRGB": 11, "xBGR": 12,       # same paths as RGBA / BGRA / ARGB / ABGR
    "Y42B": 13, "Y444": 14, "YUY2": 15, "UYVY": 16, "GRAY8": 17, "NV16": 18, "NV24": 19,
    "NV61": 20, "YVYU": 21, "VYUY": 22, "v308": 23, "IYU2": 24, "RGB": 25, "BGR": 26,
}
FLAG_PREMULTIPLIED_ALPHA = 1
MAX_RECTANGLES = 64

OK = 0
ERROR_INVALID_ARGUMENT = -1
ERROR_NO_DEVICE = -2
ERROR_CUDA = -3
ERROR_OUT_OF_MEMORY = -4
ERROR_UNSUPPORTED_FORMAT = -5
ERROR_NOT_FOUND = -6
ERROR_TOO_MANY_RECTANGLES = -7


class Rect(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32)]


class Rectangle(C.Structure):
    _fields_ = [("pixels", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32),
                ("stride", C.c_int32), ("x", C.c_int32), ("y", C.c_int32),
                ("global_alpha", C.c_float), ("flags", C.c_uint32),
                ("render_width", C.c_int32), ("render_height", C.c_int32)]


class Region(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32),
                ("background_color", C.c_uint32), ("opacity", C.c_double),
                ("layer", C.c_void_p), ("layer_stride", C.c_int32)]


class Frame(C.Structure):
    _fields_ = [("plane", C.c_void_p * 3), ("stride", C.c_int32 * 3)]


class Stats(C.Structure):
    _fields_ = [("frames_blended", C.c_uint64), ("launches", C.c_uint64),
                ("group_launches", C.c_uint64), ("prepare_launches", C.c_uint64), ("overlays_set", C.c_uint64),
                ("algorithmic_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("kernel_ms", C.c_double),
                ("kernel_ms_launches", C.c_uint64), ("cache_bytes", C.c_uint64),
                ("multi_launches", C.c_uint64), ("lazy_launches", C.c_uint64),
                ("host_dma_batches", C.c_uint64), ("opaque_skip_launches", C.c_uint64), ("staged_frames", C.c_uint64),
                ("overlays_updated", C.c_uint64), ("dependent_launches", C.c_uint64)]


# name -> (restype, argtypes); also the list tests check against the header
PROTOTYPES = {
    "fluc_ttmlblend_new": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "fluc_ttmlblend_free": (None, [C.c_void_p]),
    "fluc_ttmlblend_strerror": (C.c_char_p, [C.c_int]),
    "fluc_ttmlblend_last_cuda_error": (C.c_char_p, [C.c_void_p]),
    "fluc_ttmlblend_device_count": (C.c_int, []),
    "fluc_ttmlblend_numa_node": (C.c_int, [C.c_void_p]),
    "fluc_ttmlblend_version": (C.c_char_p, []),
    "fluc_ttmlblend_multi_new": (C.c_int, [C.POINTER(C.c_int), C.c_uint32, C.POINTER(C.c_void_p)]),
    "fluc_ttmlblend_multi_free": (None, [C.c_void_p]),
    "fluc_ttmlblend_multi_size": (C.c_uint32, [C.c_void_p]),
    "fluc_ttmlblend_multi_context": (C.c_void_p, [C.c_void_p, C.c_uint32]),
    "fluc_ttmlblend_multi_device": (C.c_int, [C.c_void_p, C.c_uint32]),
    "fluc_ttmlblend_multi_sync": (C.c_int, [C.c_void_p]),
    "fluc_ttmlblend_multi_stats_copy": (None, [C.c_void_p, C.POINTER(Stats)]),
    "fluc_ttmlblend_overlay_set": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_int32,
                                             C.c_int32, C.c_int32, C.POINTER(Rect), C.c_uint32]),
    "fluc_ttmlblend_overlay_update": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_int32,
                                                C.c_int32, C.c_int32, C.POINTER(Rect), C.c_uint32]),
    "fluc_ttmlblend_overlay_set_rectangles": (C.c_int, [C.c_void_p, C.c_uint32,
                                                        C.POINTER(Rectangle), C.c_uint32]),
    "fluc_ttmlblend_overlay_set_regions": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int32, C.c_int32,
                                                     C.POINTER(Region), C.c_uint32]),
    "fluc_ttmlblend_overlay_clear": (C.c_int, [C.c_void_p, C.c_uint32]),
    "fluc_ttmlblend_overlay_set_global_alpha": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_float),
                                                          C.c_uint32]),
    "fluc_ttmlblend_overlay_set_positions": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_int32),
                                                       C.POINTER(C.c_int32), C.c_uint32]),
    "fluc_ttmlblend_overlay_set_render_rectangles": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(Rect),
                                                               C.c_uint32]),
    "fluc_ttmlblend_set_chroma_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "fluc_ttmlblend_submit": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_int32, C.c_int32,
                                        C.c_uint32, C.POINTER(Frame), C.POINTER(Frame),
                                        C.POINTER(C.c_uint64)]),
    "fluc_ttmlblend_submit_many": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_int,
                                             C.c_int32, C.c_int32, C.c_uint32, C.POINTER(Frame),
                                             C.POINTER(Frame), C.POINTER(C.c_uint64)]),
    "fluc_ttmlblend_submit_many_repeat": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_int,
                                                    C.c_int32, C.c_int32, C.c_uint32, C.POINTER(Frame),
                                                    C.POINTER(Frame), C.c_uint32, C.c_uint32]),
    "fluc_ttmlblend_submit_many_after": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                                                   C.c_int, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(Frame),
                                                   C.POINTER(Frame), C.POINTER(C.c_uint64)]),
    "fluc_ttmlblend_wait_on_stream": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p]),
    "fluc_ttmlblend_pcie_probe": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_double, C.POINTER(C.c_double)]),
    "fluc_ttmlblend_flush": (C.c_int, [C.c_void_p]),
    "fluc_ttmlblend_wait": (C.c_int, [C.c_void_p, C.c_uint64]),
    "fluc_ttmlblend_sync": (C.c_int, [C.c_void_p]),
    "fluc_ttmlblend_set_batch": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "fluc_ttmlblend_blend_host": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_int32, C.c_int32,
                                            C.c_uint32, C.POINTER(Frame), C.POINTER(C.c_uint64)]),
    "fluc_ttmlblend_blend_host_many": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_int,
                                                 C.c_int32, C.c_int32, C.c_uint32, C.POINTER(Frame),
                                                 C.POINTER(C.c_uint64)]),
    "fluc_ttmlblend_set_auto_register": (C.c_int, [C.c_void_p, C.c_int]),
    "fluc_ttmlblend_set_host_dma": (C.c_int, [C.c_void_p, C.c_int]),
    "fluc_ttmlblend_host_register": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "fluc_ttmlblend_host_unregister": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fluc_ttmlblend_host_forget": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "fluc_ttmlblend_frame_pool_acquire": (C.c_int, [C.c_void_p, C.c_int, C.c_int32, C.c_int32,
                                                    C.c_int, C.POINTER(Frame)]),
    "fluc_ttmlblend_frame_pool_release": (C.c_int, [C.c_void_p, C.POINTER(Frame)]),
    "fluc_ttmlblend_frame_upload": (C.c_int, [C.c_void_p, C.c_int, C.c_int32, C.c_int32,
                                              C.POINTER(Frame), C.POINTER(Frame)]),
    "fluc_ttmlblend_frame_download": (C.c_int, [C.c_void_p, C.c_int, C.c_int32, C.c_int32,
                                                C.POINTER(Frame), C.POINTER(Frame)]),
    "fluc_ttmlblend_blur_argb32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                             C.c_int32, C.c_double, C.c_void_p, C.c_int32]),
    "fluc_ttmlblend_format_planes": (C.c_int, [C.c_int]),
    "fluc_ttmlblend_plane_row_bytes": (C.c_int, [C.c_int, C.c_int, C.c_int32]),
    "fluc_ttmlblend_plane_rows": (C.c_int, [C.c_int, C.c_int, C.c_int32]),
    "fluc_ttmlblend_stats_copy": (None, [C.c_void_p, C.POINTER(Stats)]),
    "fluc_ttmlblend_stats_reset": (None, [C.c_void_p]),
    "fluc_ttmlblend_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "fluc_ttmlblend_timer_begin": (C.c_int, [C.c_void_p]),
    "fluc_ttmlblend_timer_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "fluc_ttmlblend_scrub_l2": (C.c_int, [C.c_void_p, C.c_size_t]),
    "fluc_ttmlblend_stream_handle": (C.c_void_p, [C.c_void_p]),
}

_lib = None


class TtmlBlendError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str = ""):
        self.code = code
        super().__init__(f"{what}: {code} ({detail})" if detail else f"{what}: {code}")


def load_library(path: Optional[str] = None):
    """Loads the C-ABI library. Fails loudly if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("FLUC_TTMLBLEND_LIB") or LIB_PATH   # env: kernel-variant experiments
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} is missing: build it with `make -C {os.path.dirname(p)}` "
            "(or __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(p)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def plane_layout(fmt: str, width: int, height: int):
    """[(row_bytes, rows)] per plane, as GStreamer lays the format out."""
    f = fmt.upper()
    if f in ("I420", "YV12"):
        cw, ch = (width + 1) // 2, (height + 1) // 2
        return [(width, height), (cw, ch), (cw, ch)]
    if f in ("NV12", "NV21"):
        cw, ch = (width + 1) // 2, (height + 1) // 2
        return [(width, height), (2 * cw, ch)]
    if f in ("NV16", "NV61"):
        return [(width, height), (2 * ((width + 1) // 2), height)]
    if f == "NV24":
        return [(width, height), (2 * width, height)]
    if f == "Y42B":
        return [(width, height), ((width + 1) // 2, height), ((width + 1) // 2, height)]
    if f == "Y444":
        return [(width, height)] * 3
    if f in ("YUY2", "UYVY", "YVYU", "VYUY"):
        return [(4 * ((width + 1) // 2), height)]
    if f in ("V308", "IYU2", "RGB", "BGR"):
        return [(3 * width, height)]
    if f == "GRAY8":
        return [(width, height)]
    return [(4 * width, height)]


def frame_bytes(fmt: str, width: int, height: int) -> int:
    return sum(rb * r for rb, r in plane_layout(fmt, width, height))


def _frame_from_arrays(planes: Sequence[np.ndarray]) -> Frame:
    f = Frame()
    for i, p in enumerate(planes):
        assert p.dtype == np.uint8 and p.ndim == 2 and p.strides[1] == 1
        f.plane[i] = p.ctypes.data
        f.stride[i] = p.strides[0]
    return f


class DeviceFrame:
    """A pool frame in HBM (or pinned host memory when on_host)."""

    def __init__(self, ctx: "TtmlBlend", fmt: str, width: int, height: int, on_host: bool = False):
        self.ctx, self.fmt, self.width, self.height, self.on_host = ctx, fmt, width, height, on_host
        self.c = Frame()
        ctx._check(ctx.lib.fluc_ttmlblend_frame_pool_acquire(
            ctx.h, FORMATS[fmt], width, height, 1 if on_host else 0, C.byref(self.c)), "frame_pool_acquire")
        self._released = False

    def release(self):
        if not self._released:
            self._released = True
            self.ctx._check(self.ctx.lib.fluc_ttmlblend_frame_pool_release(self.ctx.h, C.byref(self.c)),
                            "frame_pool_release")

    def host_planes(self):
        """numpy views of a pinned host frame's planes (on_host only)."""
        assert self.on_host
        out = []
        for i, (rb, rows) in enumerate(plane_layout(self.fmt, self.width, self.height)):
            stride = self.c.stride[i]
            buf = (C.c_uint8 * (stride * rows)).from_address(self.c.plane[i])
            out.append(np.frombuffer(buf, dtype=np.uint8).reshape(rows, stride)[:, :rb])
        return out

    def upload(self, planes: Sequence[np.ndarray]):
        src = _frame_from_arrays(planes)
        self.ctx._check(self.ctx.lib.fluc_ttmlblend_frame_upload(
            self.ctx.h, FORMATS[self.fmt], self.width, self.height, C.byref(src), C.byref(self.c)),
            "frame_upload")

    def download(self):
        planes = [np.zeros((rows, rb), dtype=np.uint8)
                  for rb, rows in plane_layout(self.fmt, self.width, self.height)]
        dst = _frame_from_arrays(planes)
        self.ctx._check(self.ctx.lib.fluc_ttmlblend_frame_download(
            self.ctx.h, FORMATS[self.fmt], self.width, self.height, C.byref(self.c), C.byref(dst)),
            "frame_download")
        return planes


class TtmlBlend:
    """One context per GPU (FlucTtmlBlend)."""

    def __init__(self, device: int = 0, lib_path: Optional[str] = None, _borrowed=None):
        self.lib = load_library(lib_path)
        self._owned = _borrowed is None
        if _borrowed is not None:               # a context owned by a TtmlBlendMulti
            self.h = C.c_void_p(_borrowed)
            return
        self.h = C.c_void_p()
        rc = self.lib.fluc_ttmlblend_new(device, C.byref(self.h))
        if rc != OK:
            self.h = None
            raise TtmlBlendError(rc, "fluc_ttmlblend_new", self.lib.fluc_ttmlblend_strerror(rc).decode())

    def close(self):
        if getattr(self, "h", None):
            if self._owned:
                self.lib.fluc_ttmlblend_free(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != OK:
            detail = self.lib.fluc_ttmlblend_strerror(rc).decode()
            cuda = self.lib.fluc_ttmlblend_last_cuda_error(self.h).decode() if self.h else ""
            raise TtmlBlendError(rc, what, f"{detail}; {cuda}" if cuda else detail)

    def numa_node(self) -> int:
        return self.lib.fluc_ttmlblend_numa_node(self.h)

    # -- overlay cache ---------------------------------------------------
    def overlay_set(self, stream: int, bgra: np.ndarray, rects: Iterable[Sequence[int]] = ()):
        """ttmlrender form: H x W x 4 premultiplied BGRA image + region boxes (x, y, w, h)."""
        assert bgra.dtype == np.uint8 and bgra.ndim == 3 and bgra.shape[2] == 4 and bgra.strides[2] == 1
        rl = list(rects)
        arr = (Rect * max(1, len(rl)))(*[Rect(*map(int, r)) for r in rl])
        self._check(self.lib.fluc_ttmlblend_overlay_set(
            self.h, stream, bgra.ctypes.data, bgra.shape[1], bgra.shape[0], bgra.strides[0],
            arr if rl else None, len(rl)), "overlay_set")

    def overlay_update(self, stream: int, bgra: np.ndarray, changed: Iterable[Sequence[int]]):
        """The next state of the stream's cue: the new H x W x 4 image and the boxes (x, y, w, h)
        outside which it equals the previous one. Untouched regions keep their prepared planes."""
        assert bgra.dtype == np.uint8 and bgra.ndim == 3 and bgra.shape[2] == 4 and bgra.strides[2] == 1
        rl = list(changed)
        arr = (Rect * max(1, len(rl)))(*[Rect(*map(int, r)) for r in rl])
        self._check(self.lib.fluc_ttmlblend_overlay_update(
            self.h, stream, bgra.ctypes.data, bgra.shape[1], bgra.shape[0], bgra.strides[0],
            arr if rl else None, len(rl)), "overlay_update")

    def overlay_set_rectangles(self, stream: int, rectangles: Sequence[dict]):
        """GstVideoOverlayComposition form. Each dict: pixels (h x w x 4 uint8 BGRA), x, y,
        global_alpha (default 1.0), premultiplied (default True), render_width / render_height
        (default: the pixel size; anything else is scaled like GStreamer does before blending)."""
        n = len(rectangles)
        arr = (Rectangle * max(1, n))()
        for i, r in enumerate(rectangles):
            px = r["pixels"]
            assert px.dtype == np.uint8 and px.ndim == 3 and px.shape[2] == 4 and px.strides[2] == 1
            arr[i] = Rectangle(px.ctypes.data, px.shape[1], px.shape[0], px.strides[0],
                               int(r.get("x", 0)), int(r.get("y", 0)),
                               float(r.get("global_alpha", 1.0)),
                               FLAG_PREMULTIPLIED_ALPHA if r.get("premultiplied", True) else 0,
                               int(r.get("render_width", 0)), int(r.get("render_height", 0)))
        self._check(self.lib.fluc_ttmlblend_overlay_set_rectangles(self.h, stream, arr, n),
                    "overlay_set_rectangles")

    def overlay_set_regions(self, stream: int, width: int, height: int, regions: Sequence[dict]):
        """Region form: the overlay is composed on the GPU. Each dict: x, y, w, h,
        background_color (0xRRGGBBAA), opacity, layer (h x w x 4 uint8 premultiplied BGRA or None)."""
        n = len(regions)
        arr = (Region * max(1, n))()
        for i, r in enumerate(regions):
            layer = r.get("layer")
            if layer is not None:
                assert layer.dtype == np.uint8 and layer.shape == (r["h"], r["w"], 4) and layer.strides[2] == 1
            arr[i] = Region(r["x"], r["y"], r["w"], r["h"], r.get("background_color", 0),
                            float(r.get("opacity", 1.0)),
                            layer.ctypes.data if layer is not None else None,
                            layer.strides[0] if layer is not None else 0)
        self._check(self.lib.fluc_ttmlblend_overlay_set_regions(self.h, stream, width, height, arr, n),
                    "overlay_set_regions")

    def overlay_clear(self, stream: int):
        self._check(self.lib.fluc_ttmlblend_overlay_clear(self.h, stream), "overlay_clear")

    def overlay_set_global_alpha(self, stream: int, alphas):
        """gst_video_overlay_rectangle_set_global_alpha for the stream's current overlay, without a
        new upload or prepare. `alphas`: one float for every rectangle, or a sequence with one value
        per rectangle the overlay was installed with (overlay_set_rectangles: list order;
        overlay_set: its region boxes). Frames submitted afterwards blend with the new values."""
        vals = [float(alphas)] if np.ndim(alphas) == 0 else [float(a) for a in alphas]
        arr = (C.c_float * max(1, len(vals)))(*vals)
        self._check(self.lib.fluc_ttmlblend_overlay_set_global_alpha(self.h, stream, arr, len(vals)),
                    "overlay_set_global_alpha")

    def overlay_set_positions(self, stream: int, xs: Sequence[int], ys: Sequence[int]):
        """gst_video_overlay_rectangle_set_render_rectangle for the position only: rectangle i of
        the stream's overlay_set_rectangles list goes to (xs[i], ys[i]), without a new upload, scale
        or scan. Frames submitted afterwards blend the rectangles at their new positions."""
        xl, yl = [int(v) for v in xs], [int(v) for v in ys]
        if len(xl) != len(yl):
            raise ValueError("overlay_set_positions: xs and ys differ in length")
        ax = (C.c_int32 * max(1, len(xl)))(*xl)
        ay = (C.c_int32 * max(1, len(yl)))(*yl)
        self._check(self.lib.fluc_ttmlblend_overlay_set_positions(self.h, stream, ax, ay, len(xl)),
                    "overlay_set_positions")

    def overlay_set_render_rectangles(self, stream: int, rects: Iterable[Sequence[int]]):
        """gst_video_overlay_rectangle_set_render_rectangle: rectangle i of the stream's
        overlay_set_rectangles list is placed at (x, y) of rects[i] = (x, y, w, h) and rendered at
        w x h (0: its pixel size), scaled again on the GPU from its resident pixels, without a new
        upload. Frames submitted afterwards blend the rectangles at their new render rectangles."""
        rl = [tuple(int(v) for v in r) for r in rects]
        arr = (Rect * max(1, len(rl)))(*[Rect(*r) for r in rl])
        self._check(self.lib.fluc_ttmlblend_overlay_set_render_rectangles(self.h, stream, arr, len(rl)),
                    "overlay_set_render_rectangles")

    def set_chroma_mode(self, average: bool):
        """False (default): GStreamer's sited chroma, bit-exact. True: 2x2 mean, NOT bit-exact."""
        self._check(self.lib.fluc_ttmlblend_set_chroma_mode(self.h, 1 if average else 0), "set_chroma_mode")

    # -- device-resident frames -----------------------------------------
    def submit(self, stream: int, fmt: str, width: int, height: int, src: Frame, dst: Frame,
               frame_flags: int = 0) -> int:
        t = C.c_uint64()
        self._check(self.lib.fluc_ttmlblend_submit(
            self.h, stream, FORMATS[fmt], width, height, frame_flags, C.byref(src), C.byref(dst),
            C.byref(t)), "submit")
        return t.value

    class Batch:
        """Pre-marshalled arguments of submit_many (arrays of streams / frames / tickets)."""

        def __init__(self, streams, fmt, width, height, srcs, dsts, frame_flags=0):
            """dsts may hold several sets of len(streams) frames (submit_many_repeat rotates them)."""
            n = len(streams)
            assert len(dsts) % n == 0 and len(dsts) >= n
            self.n, self.fmt, self.width, self.height, self.flags = n, FORMATS[fmt], width, height, frame_flags
            self.dst_sets = len(dsts) // n
            self.streams = (C.c_uint32 * n)(*streams)
            self.srcs = (Frame * n)(*srcs)
            self.dsts = (Frame * len(dsts))(*dsts)
            self.tickets = (C.c_uint64 * n)()

    def submit_many(self, batch: "TtmlBlend.Batch"):
        """One C call for a whole batch; returns the ticket array (ctypes)."""
        self._check(self.lib.fluc_ttmlblend_submit_many(
            self.h, batch.n, batch.streams, batch.fmt, batch.width, batch.height, batch.flags,
            batch.srcs, batch.dsts, batch.tickets), "submit_many")
        return batch.tickets

    def submit_many_after(self, batch: "TtmlBlend.Batch", cuda_stream: int):
        """submit_many ordered after the work already enqueued on a CUDA stream of the context's
        device (the raw cudaStream_t handle, e.g. torch.cuda.current_stream().cuda_stream; 0: the
        legacy default stream). The host does not wait for that work. Returns the ticket array."""
        self._check(self.lib.fluc_ttmlblend_submit_many_after(
            self.h, cuda_stream or None, batch.n, batch.streams, batch.fmt, batch.width, batch.height,
            batch.flags, batch.srcs, batch.dsts, batch.tickets), "submit_many_after")
        return batch.tickets

    def wait_on_stream(self, ticket: int, cuda_stream: int):
        """Work enqueued on the CUDA stream after this call runs after the ticket's frame is
        complete; the host does not wait."""
        self._check(self.lib.fluc_ttmlblend_wait_on_stream(self.h, ticket, cuda_stream or None),
                    "wait_on_stream")

    def submit_many_repeat(self, batch: "TtmlBlend.Batch", repeats: int):
        """`repeats` x submit_many (+ flush) inside one C call (bench helper)."""
        self._check(self.lib.fluc_ttmlblend_submit_many_repeat(
            self.h, batch.n, batch.streams, batch.fmt, batch.width, batch.height, batch.flags,
            batch.srcs, batch.dsts, batch.dst_sets, repeats), "submit_many_repeat")

    def pcie_probe(self, mode: int, nbytes: int, seconds: float) -> float:
        """GB/s per direction PCIe carries for this GPU right now: mode 0 copy engine both ways,
        mode 1 a kernel rewriting host memory in place (bench helper)."""
        g = C.c_double()
        self._check(self.lib.fluc_ttmlblend_pcie_probe(self.h, mode, nbytes, float(seconds), C.byref(g)),
                    "pcie_probe")
        return g.value

    def flush(self):
        self._check(self.lib.fluc_ttmlblend_flush(self.h), "flush")

    def wait(self, ticket: int):
        self._check(self.lib.fluc_ttmlblend_wait(self.h, ticket), "wait")

    def sync(self):
        self._check(self.lib.fluc_ttmlblend_sync(self.h), "sync")

    def set_batch(self, max_frames: int, linger_us: int):
        self._check(self.lib.fluc_ttmlblend_set_batch(self.h, max_frames, linger_us), "set_batch")

    # -- host-resident frames: gst_video_overlay_composition_blend ------
    def blend_host(self, stream: int, fmt: str, width: int, height: int,
                   planes: Sequence[np.ndarray], frame_flags: int = 0) -> int:
        f = _frame_from_arrays(planes)
        return self.blend_host_frame(stream, fmt, width, height, f, frame_flags)

    def blend_host_frame(self, stream: int, fmt: str, width: int, height: int, frame: Frame,
                         frame_flags: int = 0) -> int:
        t = C.c_uint64()
        self._check(self.lib.fluc_ttmlblend_blend_host(
            self.h, stream, FORMATS[fmt], width, height, frame_flags, C.byref(frame), C.byref(t)),
            "blend_host")
        return t.value

    def blend_host_many(self, batch: "TtmlBlend.Batch"):
        """One C call for a batch of host frames (batch.dsts; modified in place); returns the
        ticket array."""
        self._check(self.lib.fluc_ttmlblend_blend_host_many(
            self.h, batch.n, batch.streams, batch.fmt, batch.width, batch.height, batch.flags,
            batch.dsts, batch.tickets), "blend_host_many")
        return batch.tickets

    def set_auto_register(self, on: bool):
        self._check(self.lib.fluc_ttmlblend_set_auto_register(self.h, 1 if on else 0), "set_auto_register")

    def set_host_dma(self, mode: int):
        """How batches of pinned pool frames cross PCIe: 0 zero copy, 1 copy engines, 2 measured (default)."""
        self._check(self.lib.fluc_ttmlblend_set_host_dma(self.h, int(mode)), "set_host_dma")

    def host_register(self, arr: np.ndarray):
        self._check(self.lib.fluc_ttmlblend_host_register(self.h, arr.ctypes.data, arr.nbytes),
                    "host_register")

    def host_unregister(self, arr: np.ndarray):
        self._check(self.lib.fluc_ttmlblend_host_unregister(self.h, arr.ctypes.data), "host_unregister")

    def host_forget(self, arr: np.ndarray) -> int:
        """Drops the automatic registrations inside `arr` (call before the memory is freed)."""
        n = self.lib.fluc_ttmlblend_host_forget(self.h, arr.ctypes.data, arr.nbytes)
        if n < 0:
            self._check(n, "host_forget")
        return n

    def blur_argb32(self, img: np.ndarray, radius: int, sigma: float) -> np.ndarray:
        """gst_ttml_blur_image_surface (surface, radius, sigma): h x w x 4 uint8 in and out."""
        assert img.dtype == np.uint8 and img.ndim == 3 and img.shape[2] == 4 and img.strides[2] == 1
        out = np.zeros_like(img)
        self._check(self.lib.fluc_ttmlblend_blur_argb32(
            self.h, img.ctypes.data, img.shape[1], img.shape[0], img.strides[0], radius, float(sigma),
            out.ctypes.data, out.strides[0]), "blur_argb32")
        return out

    # -- pool / stats ----------------------------------------------------
    def acquire(self, fmt: str, width: int, height: int, on_host: bool = False) -> DeviceFrame:
        return DeviceFrame(self, fmt, width, height, on_host)

    def stats(self) -> dict:
        s = Stats()
        self.lib.fluc_ttmlblend_stats_copy(self.h, C.byref(s))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def stats_reset(self):
        self.lib.fluc_ttmlblend_stats_reset(self.h)

    def set_profiling(self, every: int):
        """0 / False: off; 1 / True: time every launch; n: time every n-th launch."""
        self._check(self.lib.fluc_ttmlblend_set_profiling(self.h, int(every)), "set_profiling")

    def timer_begin(self):
        self._check(self.lib.fluc_ttmlblend_timer_begin(self.h), "timer_begin")

    def timer_end(self) -> float:
        ms = C.c_double()
        self._check(self.lib.fluc_ttmlblend_timer_end(self.h, C.byref(ms)), "timer_end")
        return ms.value

    def scrub_l2(self, nbytes: int = 256 << 20):
        self._check(self.lib.fluc_ttmlblend_scrub_l2(self.h, nbytes), "scrub_l2")


class TtmlBlendMulti:
    """Several GPUs in one process (FlucTtmlBlendMulti): stream s lives on context s % n."""

    def __init__(self, devices: Sequence[int] = ()):
        self.lib = load_library()
        self.h = C.c_void_p()
        arr = (C.c_int * max(1, len(devices)))(*devices)
        rc = self.lib.fluc_ttmlblend_multi_new(arr if devices else None, len(devices), C.byref(self.h))
        if rc != OK:
            self.h = None
            raise TtmlBlendError(rc, "fluc_ttmlblend_multi_new", self.lib.fluc_ttmlblend_strerror(rc).decode())
        self._ctx = {}

    def size(self) -> int:
        return self.lib.fluc_ttmlblend_multi_size(self.h)

    def context(self, stream: int) -> TtmlBlend:
        k = stream % self.size()
        if k not in self._ctx:
            self._ctx[k] = TtmlBlend(_borrowed=self.lib.fluc_ttmlblend_multi_context(self.h, stream))
        return self._ctx[k]

    def device(self, stream: int) -> int:
        return self.lib.fluc_ttmlblend_multi_device(self.h, stream)

    def sync(self):
        rc = self.lib.fluc_ttmlblend_multi_sync(self.h)
        if rc != OK:
            raise TtmlBlendError(rc, "fluc_ttmlblend_multi_sync", self.lib.fluc_ttmlblend_strerror(rc).decode())

    def stats(self) -> dict:
        s = Stats()
        self.lib.fluc_ttmlblend_multi_stats_copy(self.h, C.byref(s))
        return {name: getattr(s, name) for name, _ in Stats._fields_}

    def close(self):
        if getattr(self, "h", None):
            for c in self._ctx.values():
                c.h = None
            self.lib.fluc_ttmlblend_multi_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def composition_blend(ctx: TtmlBlend, stream: int, fmt: str, width: int, height: int,
                      planes: Sequence[np.ndarray], frame_flags: int = 0):
    """gst_video_overlay_composition_blend(comp, frame) on host planes, in place, synchronous."""
    ctx.wait(ctx.blend_host(stream, fmt, width, height, planes, frame_flags))
    return planes
