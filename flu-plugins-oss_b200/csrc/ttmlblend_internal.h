/*
 * ttmlblend_internal.h -- shared declarations of the host runtime behind the C ABI
 * (include/fluc_ttmlblend.h). Private to csrc/. The runtime is split by concern:
 *   overlay_cache.cu  upload, auto-crop, once-per-cue prepare, deferred frees
 *   jobs.cu           frame -> bands / windows / job classes / groups
 *   scheduler.cu      batches, table slots, launches, the scheduler thread
 *   fluc_ttmlblend.cu the extern "C" entry points (context, submit, host frames, pool, stats)
 */
#ifndef TTMLBLEND_INTERNAL_H
#define TTMLBLEND_INTERNAL_H

#include "../../include/fluc_ttmlblend.h"
#include "ttmlblend_kernels.cuh"

#include <nvtx3/nvToolsExt.h>       /* header-only: ranges show up in nsys / ncu timelines */

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace tbh {

using namespace tb;

/* ---------------------------------------------------------------------- */
/* format geometry                                                        */

/* RGBx / BGRx / xRGB / xBGR -> RGBA / BGRA / ARGB / ABGR (same pack/unpack in GStreamer) */
inline int
format_canon (int f)
{
  switch (f) {
    case FLUC_TTMLBLEND_FORMAT_RGBx: return FLUC_TTMLBLEND_FORMAT_RGBA;
    case FLUC_TTMLBLEND_FORMAT_BGRx: return FLUC_TTMLBLEND_FORMAT_BGRA;
    case FLUC_TTMLBLEND_FORMAT_xRGB: return FLUC_TTMLBLEND_FORMAT_ARGB;
    case FLUC_TTMLBLEND_FORMAT_xBGR: return FLUC_TTMLBLEND_FORMAT_ABGR;
    default: return f;
  }
}

inline bool
format_valid (int f)
{
  return f >= 0 && f < FLUC_TTMLBLEND_FORMAT_COUNT;
}

/* chroma subsampling of the planar / semi-planar YUV formats (1 = none) */
inline int
format_sub_x (int f)
{
  switch (f) {
    case FLUC_TTMLBLEND_FORMAT_I420:
    case FLUC_TTMLBLEND_FORMAT_YV12:
    case FLUC_TTMLBLEND_FORMAT_NV12:
    case FLUC_TTMLBLEND_FORMAT_NV21:
    case FLUC_TTMLBLEND_FORMAT_Y42B:
    case FLUC_TTMLBLEND_FORMAT_NV16:
    case FLUC_TTMLBLEND_FORMAT_NV61:
      return 2;
    default:
      return 1;
  }
}

inline int
format_sub_y (int f)
{
  switch (f) {
    case FLUC_TTMLBLEND_FORMAT_I420:
    case FLUC_TTMLBLEND_FORMAT_YV12:
    case FLUC_TTMLBLEND_FORMAT_NV12:
    case FLUC_TTMLBLEND_FORMAT_NV21:
      return 2;
    default:
      return 1;
  }
}

inline bool
format_packed_422 (int f)
{
  return f == FLUC_TTMLBLEND_FORMAT_YUY2 || f == FLUC_TTMLBLEND_FORMAT_UYVY ||
      f == FLUC_TTMLBLEND_FORMAT_YVYU || f == FLUC_TTMLBLEND_FORMAT_VYUY;
}

/* packed 4:4:4 with three bytes per pixel (no alpha byte) */
inline bool
format_packed_444_3 (int f)
{
  return f == FLUC_TTMLBLEND_FORMAT_v308 || f == FLUC_TTMLBLEND_FORMAT_IYU2;
}

inline int
format_planes (int f)
{
  switch (f) {
    case FLUC_TTMLBLEND_FORMAT_I420:
    case FLUC_TTMLBLEND_FORMAT_YV12:
    case FLUC_TTMLBLEND_FORMAT_Y42B:
    case FLUC_TTMLBLEND_FORMAT_Y444:
      return 3;
    case FLUC_TTMLBLEND_FORMAT_NV12:
    case FLUC_TTMLBLEND_FORMAT_NV21:
    case FLUC_TTMLBLEND_FORMAT_NV16:
    case FLUC_TTMLBLEND_FORMAT_NV61:
    case FLUC_TTMLBLEND_FORMAT_NV24:
      return 2;
    default:
      return 1;
  }
}

inline int
plane_row_bytes (int f, int plane, int w)
{
  switch (f) {
    case FLUC_TTMLBLEND_FORMAT_I420:
    case FLUC_TTMLBLEND_FORMAT_YV12:
    case FLUC_TTMLBLEND_FORMAT_Y42B:
      return plane == 0 ? w : (w + 1) / 2;
    case FLUC_TTMLBLEND_FORMAT_NV12:
    case FLUC_TTMLBLEND_FORMAT_NV21:
    case FLUC_TTMLBLEND_FORMAT_NV16:
    case FLUC_TTMLBLEND_FORMAT_NV61:
      return plane == 0 ? w : 2 * ((w + 1) / 2);
    case FLUC_TTMLBLEND_FORMAT_NV24:
      return plane == 0 ? w : 2 * w;
    case FLUC_TTMLBLEND_FORMAT_Y444:
    case FLUC_TTMLBLEND_FORMAT_GRAY8:
      return w;
    case FLUC_TTMLBLEND_FORMAT_YUY2:
    case FLUC_TTMLBLEND_FORMAT_UYVY:
    case FLUC_TTMLBLEND_FORMAT_YVYU:
    case FLUC_TTMLBLEND_FORMAT_VYUY:
      return 4 * ((w + 1) / 2);     /* whole macropixels */
    case FLUC_TTMLBLEND_FORMAT_v308:
    case FLUC_TTMLBLEND_FORMAT_IYU2:
    case FLUC_TTMLBLEND_FORMAT_RGB:
    case FLUC_TTMLBLEND_FORMAT_BGR:
      return 3 * w;
    default:
      return 4 * w;
  }
}

inline int
plane_rows (int f, int plane, int h)
{
  return (plane > 0 && format_sub_y (f) == 2) ? (h + 1) / 2 : h;
}

inline int
plane_kind (int f)
{
  switch (f) {
    case FLUC_TTMLBLEND_FORMAT_AYUV:
    case FLUC_TTMLBLEND_FORMAT_ARGB:
    case FLUC_TTMLBLEND_FORMAT_ABGR:
      return PK_PACKED_A0;
    case FLUC_TTMLBLEND_FORMAT_RGBA:
    case FLUC_TTMLBLEND_FORMAT_BGRA:
      return PK_PACKED_A3;
    case FLUC_TTMLBLEND_FORMAT_RGB:
    case FLUC_TTMLBLEND_FORMAT_BGR:
      return PK_PLANE8_RGB;
    default:
      return PK_PLANE8;
  }
}

inline int ceil_div (int a, int b) { return (a + b - 1) / b; }
inline size_t align_up (size_t v, size_t a) { return (v + a - 1) / a * a; }

/* Byte ranges of the frames queued in `pending`, for the hazard check of submit / blend_host:
 * sorted, disjoint, touching ranges merged. A flat vector -- a batch holds at most a few hundred
 * frames and the planes of one frame are usually neighbours, so an insert is a binary search
 * plus a short memmove, and nothing is allocated once the vector has grown. */
struct IntervalSet {
  std::vector<std::pair<uintptr_t, uintptr_t>> v;      /* [lo, hi) */
  void clear () { v.clear (); }
  bool empty () const { return v.empty (); }
  /* first range that ends after lo */
  size_t first_after (uintptr_t lo) const
  {
    size_t a = 0, b = v.size ();
    while (a < b) {
      const size_t m = (a + b) / 2;
      if (v[m].second > lo) b = m; else a = m + 1;
    }
    return a;
  }
  bool overlaps (uintptr_t lo, uintptr_t hi) const
  {
    if (v.empty () || hi <= v.front ().first || lo >= v.back ().second)
      return false;
    const size_t i = first_after (lo);
    return i < v.size () && v[i].first < hi;
  }
  void merge (const IntervalSet &o)
  {
    for (const auto &r : o.v)
      add (r.first, r.second);
  }
  void add (uintptr_t lo, uintptr_t hi)
  {
    if (hi <= lo)
      return;
    /* ranges that overlap or touch [lo, hi): those ending at or after lo and starting at or before hi */
    size_t a = 0, b = v.size ();
    while (a < b) {
      const size_t m = (a + b) / 2;
      if (v[m].second >= lo) b = m; else a = m + 1;
    }
    size_t e = a;
    while (e < v.size () && v[e].first <= hi) {
      lo = std::min (lo, v[e].first);
      hi = std::max (hi, v[e].second);
      e++;
    }
    if (e == a) {
      v.insert (v.begin () + a, std::make_pair (lo, hi));
    } else {
      v[a] = std::make_pair (lo, hi);
      v.erase (v.begin () + a + 1, v.begin () + e);
    }
  }
};

/* ---------------------------------------------------------------------- */
/* overlay cache                                                          */

struct Ctx;

/* One stream-ordered device allocation of the overlay cache, shared by whoever points into it:
 * a cue update keeps the untouched regions' pixels and prepared planes and both the old and the
 * new overlay hold them. Freed (deferred, after a fence on every stream) with its last holder. */
struct DevBlock {
  Ctx *ctx = nullptr;
  void *ptr = nullptr;
  ~DevBlock ();
};

/* device copy of one rectangle's BGRA pixels: (x, y) is the frame position of its pixel (0,0).
 * Clipped at the left / top for the ttmlrender and region forms; the composition form keeps the
 * whole rectangle, so x and y may be negative (overlay_set_positions) */
struct RawRect {
  std::shared_ptr<DevBlock> block;     /* the allocation `dev` points into */
  uint8_t *dev = nullptr;
  int pitch = 0, w = 0, h = 0;
  int x = 0, y = 0;
  int ga = 255;                        /* global alpha the prepare folds into PLANE8 alpha bytes (255 after a fade) */
  bool premul = true;
};

struct StageSpan { int plane, b0, nb, y0, rows; };       /* rows [y0, y0+rows), bytes [b0, b0+nb) of a plane */

/* The work of one frame minus its pointers: windows, classes, band list. It depends on the
 * prepared overlay, the strides, the alignment of the planes, in place or not and the frame
 * flags -- not on which buffer the frame is in -- so it is built once and shared by every
 * frame that matches (consecutive frames of a stream, pool buffers). `id` is unique per
 * context: equal id == equal band list, which is what grouping compares. */
struct Layout {
  uint64_t id = 0;
  int kind = 0;
  /* key */
  int32_t src_pitch[3] = { 0, 0, 0 }, dst_pitch[3] = { 0, 0, 0 };
  uint32_t aligned_mask = 0;           /* bit p: plane p's pointers and strides are 16-byte aligned */
  bool windowed = false;
  uint32_t frame_flags = 0;
  /* value */
  std::vector<PlaneJob> jobs;          /* table-kernel jobs, src / dst patched per frame */
  std::vector<PlaneJob> gjobs;         /* the band list's windows as table jobs (group dissolved, no room) */
  bool grouped = false;
  std::vector<BandDesc> bands;
  uint32_t chunks_per_frame = 0;
  int32_t rect_off[3] = { 0, 0, 0 };
  int32_t gflags = 0;
  const RectRef *rects_all = nullptr;
  uint64_t algo_bytes = 0;
  uint64_t window_bytes = 0;           /* bytes of all windows (what a zero-copy host frame moves each way) */
  /* host DMA batches: the rows the windows touch (neighbouring bands merged), and whether they
   * are (nearly) full rows, so that a window's rows are one contiguous run of bytes */
  mutable std::vector<StageSpan> spans;
  mutable int dma_ok = -1;             /* -1: not looked at yet */
};

/* what one rectangle of the overlay looks like from the planes of one destination format */
struct PreparedRect {
  std::vector<std::shared_ptr<DevBlock>> blocks;      /* alpha / colour planes or pixel words */
  struct { int plane; RectRef ref; } refs[3];
  int n_refs = 0;
  /* chroma_average: the averaged 4:2:0 chroma refs (planes 1, 2) have the box's global alpha
   * folded in, since the 2x2 mean weights colours by asrc (BLENDSPEC section 7). A fade prepares
   * them again on their own, so their planes are kept apart from the luma's. */
  std::vector<std::shared_ptr<DevBlock>> avg_blocks;
  int avg_ga = -1;                     /* the global alpha folded into them; -1: no averaged chroma */
};

/* everything frame-independent, for one (format, W, H) */
struct Prepared {
  int format = -1, W = 0, H = 0;
  bool chroma_average = false;         /* prepared with the non-parity 2x2 chroma mean */
  std::vector<PreparedRect> per_rect;  /* one per Overlay::rects entry, same order */
  std::shared_ptr<DevBlock> table_block;              /* the RectRef tables */
  std::vector<RectRef> h_rects[3];     /* per plane, host copy */
  std::vector<RectRef> h_rects_all;
  RectRef *d_rects[3] = { nullptr, nullptr, nullptr };
  RectRef *d_rects_all = nullptr;      /* the three tables, contiguous */
  int32_t rect_off[3] = { 0, 0, 0 };   /* first entry of plane p in d_rects_all */
  uint64_t overlay_px = 0;             /* sum of clipped w*h */
  bool fade = false;                   /* a RectRef has a_ga != 255: launches holding it take the JF_GA variant */
  std::vector<PrepareItem> h_items;    /* a move's batch prepare items, when uploaded (source of the async copy) */
  cudaEvent_t ready = nullptr;
  bool blend_waited = false;           /* blend stream already ordered after `ready` */
  bool used = false;                   /* a frame has been blended with it (worth preparing the next cue for) */
  std::vector<std::unique_ptr<Layout>> layouts;
  ~Prepared ();                        /* destroys `ready` when set */
};

/* The pixels a rectangle of the composition form was installed from, whole and at their pixel
 * size: the rectangle's raw block when it was installed unscaled, its own block otherwise.
 * overlay_set_render_rectangles scales (or scans) them again for a new render size. */
struct BoxSource {
  std::shared_ptr<DevBlock> block;
  const uint8_t *dev = nullptr;
  int pitch = 0, w = 0, h = 0;
  bool premul = true;
};

/* One rectangle as it was handed in (a region box of ttmlrender's image): the unit a cue update
 * keeps or replaces. */
struct OverlayBox {
  FlucTtmlBlendRect declared = { 0, 0, 0, 0 };       /* frame coordinates (clipped at the left / top but for the composition form) */
  uint32_t first_rect = 0, n_rects = 0;              /* its cropped sub-rectangles in Overlay::rects */
  uint64_t groups_all = 0, groups_on = 0, groups_opaque = 0;   /* 16-pixel groups under them: all / some alpha / alpha 255 */
  int ga = 255;                        /* its current global alpha (overlay_set_global_alpha) */
  uint32_t slot = 0;                   /* which value of overlay_set_global_alpha's list is its own */
  BoxSource src;                       /* composition form only; declared.w / h are its render size */
};

struct Overlay {
  Ctx *ctx = nullptr;
  std::vector<RawRect> rects;          /* what gets prepared: cropped to non-transparent pixels */
  std::vector<OverlayBox> boxes;
  std::vector<FlucTtmlBlendRect> declared;   /* rectangles as handed in (algorithmic bytes) */
  /* ttmlrender form (overlay_set): one w x h image at the frame's origin, premultiplied, global
   * alpha 1 -- what overlay_update can patch */
  int image_w = 0, image_h = 0;
  bool updatable = false;
  bool movable = false;                /* composition form (overlay_set_rectangles): overlay_set_positions takes it */
  uint32_t n_alphas = 1;               /* global alphas overlay_set_global_alpha takes besides one for all */
  std::vector<std::unique_ptr<Prepared>> prepared;
  double transparent_fraction = 0.0;   /* of the 16-pixel groups under the kept rectangles */
  double opaque_fraction = 0.0;        /* alpha 255 all over (and the box's global alpha 1) */
  bool lazy_inplace = false;           /* in-place group launches look at the overlay first */
  bool opaque_skip = false;            /* out-of-place group launches do: no frame read under opaque vectors */
  ~Overlay ();
};

/* The event submit_many_after records on the caller's stream, shared by every frame of the call.
 * The first launch that carries one of them orders the blend stream after it (or finds it already
 * complete); later launches follow in stream order. Back to the event pool with its last frame.
 * Destroyed under the context lock. */
struct StreamAfter {
  Ctx *ctx = nullptr;
  cudaEvent_t ev = nullptr;
  bool resolved = false;               /* the blend stream is ordered after it */
  ~StreamAfter ();
};

struct PendingFrame {
  uint64_t ticket;
  uint32_t stream;
  bool host = false;                   /* a device-accessible HOST frame, blended in place (zero copy or DMA batch) */
  uintptr_t host_lo = 0, host_hi = 0;  /* its bytes (hull of the planes) */
  std::shared_ptr<StreamAfter> after;  /* submit_many_after: the caller's work to wait for */
  std::shared_ptr<Overlay> overlay;    /* keeps prep and layout alive */
  Prepared *prep;
  const Layout *layout;
  const uint8_t *src[3];
  uint8_t *dst[3];
};

/* frames that can share one launch: everything but the pointers is equal */
struct Group {
  int kind;
  uint64_t layout_id;
  bool dissolved;                      /* too small to be worth a launch: frames go to the table kernel */
  GroupParams P;
  Group () {}                          /* user-provided: no zeroing of the 19.5 KB block per launch (group_start fills in what is used) */
};

/* frames of one kind / pitch set / flag set with different band lists, packed into one
 * multi-layout launch; layouts = (first band, number of bands) of the distinct lists so far */
struct MultiGroup {
  int kind = 0;
  uint32_t n_bands = 0;
  struct Slot { uint64_t id; uint16_t band0, n_bands; };
  std::vector<Slot> layouts;
  MultiParams P;
};

/* a group launch below this many chunks (16 KB each; 4096 = 64 MB, ~10 us of HBM time) is
 * dissolved when there is a table launch to join */
constexpr uint32_t kMinGroupChunks = 4096;

struct Batch {
  uint64_t last_ticket;
  cudaEvent_t done;
  cudaEvent_t t0, t1;                  /* profiling pair (may be null) */
  std::vector<std::shared_ptr<Overlay>> keep;
  bool dma = false;                    /* host frames moved by the copy engines: `done` is on the copy-out stream */
  IntervalSet host_ranges;             /* the host frames of the batch (zero copy or DMA), for ordering later DMA batches */
  cudaEvent_t ev_in = nullptr, ev_blend = nullptr;   /* DMA batch: copy-in done, blend done (back to the pool with the batch) */
};

/* device staging for one DMA batch of host frames: full-size device frames at a constant spacing */
struct DmaSet {
  uint8_t *dev = nullptr;
  size_t bytes = 0;
  cudaEvent_t done = nullptr;          /* the copy back out of this set has finished */
  bool used = false;
};
constexpr int64_t kDmaTrialFrames = 128, kDmaSteadyFrames = 32768;   /* the first steady phases are shorter: 2048, 8192 */
constexpr int kDmaSets = 8;           /* 3 in use for whole batches, all of them for pieces (Ctx::dma_piece) */

struct TableSlot {
  PlaneJob *h_jobs = nullptr, *d_jobs = nullptr;
  uint32_t *h_begin = nullptr, *d_begin = nullptr;
  size_t cap = 0, cap_words = 0;       /* jobs / words (job begins + coarse index) */
  cudaEvent_t copied = nullptr;        /* last kernel that read the slot has finished */
  cudaEvent_t uploaded = nullptr;      /* table copy has landed */
};

/* The bytes a frame's planes occupy, as at most three ranges (planes that are neighbours in
 * memory -- pool frames, GStreamer's default layout -- come out as one). */
struct FrameExtent {
  uintptr_t lo[3], hi[3];
  int n = 0;
  FrameExtent (int fmt, int W, int H, const FlucTtmlBlendFrame *f)
  {
    for (int pl = 0; pl < format_planes (fmt); pl++) {
      const uintptr_t a = (uintptr_t) f->plane[pl];
      const uintptr_t b = a + (uintptr_t) f->stride[pl] * (uintptr_t) (plane_rows (fmt, pl, H) - 1) +
          (uintptr_t) plane_row_bytes (fmt, pl, W);
      if (n && a >= lo[n - 1] && a <= hi[n - 1] + 4096)
        hi[n - 1] = std::max (hi[n - 1], b);
      else {
        lo[n] = a;
        hi[n] = b;
        n++;
      }
    }
  }
  uintptr_t hull_lo () const
  {
    uintptr_t v = lo[0];
    for (int i = 1; i < n; i++)
      v = std::min (v, lo[i]);
    return v;
  }
  uintptr_t hull_hi () const
  {
    uintptr_t v = hi[0];
    for (int i = 1; i < n; i++)
      v = std::max (v, hi[i]);
    return v;
  }
  bool hits (const IntervalSet &s) const
  {
    for (int i = 0; i < n; i++)
      if (s.overlaps (lo[i], hi[i]))
        return true;
    return false;
  }
  void add_to (IntervalSet &s) const
  {
    for (int i = 0; i < n; i++)
      s.add (lo[i], hi[i]);
  }
};

/* do two range sets share a byte? walks the smaller one */
inline bool
sets_overlap (const IntervalSet &a, const IntervalSet &b)
{
  const IntervalSet &s = a.v.size () <= b.v.size () ? a : b, &l = a.v.size () <= b.v.size () ? b : a;
  if (s.v.empty () || l.v.empty () || s.v.back ().second <= l.v.front ().first || l.v.back ().second <= s.v.front ().first)
    return false;
  for (const auto &r : s.v)
    if (l.overlaps (r.first, r.second))
      return true;
  return false;
}

struct PoolEntry {
  void *base;                          /* slab members: the frame's first byte inside the slab */
  size_t bytes;
  bool in_slab;                        /* pinned host frames come in slabs (Ctx::host_slabs), freed with them */
  int fmt, W, H, on_host;
  FlucTtmlBlendFrame frame;
};

/* ---- staged host frames (staging.cu) ---- */
struct StageJob {
  enum State { COPY_IN, ON_GPU, COPY_OUT, DONE };
  uint64_t ticket = 0;                 /* what blend_host handed out */
  uint64_t gpu_ticket = 0;             /* the staging frame's own ticket in the batch */
  uint32_t stream = 0;
  int fmt = 0, W = 0, H = 0;
  uint32_t frame_flags = 0;
  FlucTtmlBlendFrame user = {};        /* the caller's frame */
  uintptr_t user_lo = 0, user_hi = 0;
  PoolEntry slot = {};                 /* pinned staging frame */
  std::shared_ptr<Overlay> ov;
  Prepared *prep = nullptr;
  std::vector<StageSpan> spans;
  State state = COPY_IN;
  int rc = 0;
};

constexpr int kTableSlots = 8;

struct Ctx {
  int device = 0;
  std::mutex mu;
  std::condition_variable cv;          /* wakes the scheduler thread */
  std::condition_variable launched_cv; /* a batch has been launched (waiters that let it linger) */
  /* the streams of the last submissions: with more than one active, a synchronous caller's
   * wait lets the batch linger so that other streams' frames can join its launch */
  uint32_t recent_streams[16] = {};
  uint32_t recent_pos = 0, recent_n = 0;
  int sticky = 0;
  std::string cuda_error;

  cudaStream_t blend_stream = nullptr, up_stream = nullptr, reaper = nullptr, table_stream = nullptr;
  cudaMemPool_t mem_pool = nullptr;    /* stream-ordered allocations of the overlay cache */
  cudaEvent_t ev_fence[2] = {};        /* free_deferred: blend_stream, up_stream */
  cudaEvent_t timer0 = nullptr, timer1 = nullptr;

  std::unordered_map<uint32_t, std::shared_ptr<Overlay>> overlays;
  /* layouts of frames without an overlay (pass-through copies), by format / size */
  struct BareLayouts { int format, W, H; std::vector<std::unique_ptr<Layout>> layouts; };
  std::vector<BareLayouts> bare_layouts;
  uint64_t next_layout_id = 0;
  /* band lists seen so far, by hash: layouts of different overlays (streams) with the same
   * bands, strides and flags get the same id and so share group launches */
  struct LayoutSig { uint64_t id; int kind; int32_t gflags; int32_t pitch[6], rect_off[3]; std::vector<BandDesc> bands; };
  std::unordered_map<uint64_t, std::vector<LayoutSig>> layout_sigs;
  size_t n_layout_sigs = 0;

  std::vector<PendingFrame> pending;
  std::vector<Group> groups;           /* scratch of launch_pending */
  std::vector<PlaneJob> by_kind[kPlaneKinds * 2];   /* scratch: table jobs per (kind, fast) */
  std::vector<std::vector<std::shared_ptr<Overlay>>> keep_pool;   /* recycled Batch::keep vectors */
  std::vector<int> frame_group;        /* scratch: pending frame -> index into groups */
  std::vector<std::unique_ptr<MultiGroup>> multis;   /* scratch: multi-layout launches (reused) */
  /* what the frames queued in `pending` write and read: a frame that would write something a
   * queued frame writes or reads, or read something a queued frame writes, must not share their
   * launch (CTAs of one launch run in no order) -- the batch is launched first */
  IntervalSet pending_dst, pending_src;
  IntervalSet inflight_host;           /* host frames of zero-copy batches that have not been reaped yet */
  /* programmatic dependent launch: what the batches launched since the last dependent (fully
   * ordered) launch write and read; a new batch that conflicts with them is launched JF_DEP */
  IntervalSet inflight_dst, inflight_src;
  bool use_pdl = true;                 /* FLUC_TTMLBLEND_PDL=0: ordinary, serialised launches */
  bool isolate_next = false;           /* the launch after a timed one must not overlap it */
  /* the blend stream has been told to wait for an event since the last launch: the next launch
   * goes out as an ordinary one. A programmatic launch behind a stream wait holds back the
   * completion of what was recorded before the wait (measured: a copy-out gated by an event
   * after kernel i did not start until the copy-in that kernel i+1 waits for had finished) */
  bool blend_stream_waits = false;
  /* batches whose launch failed half way (out of memory): wait() on their tickets reports it */
  struct FailedRange { uint64_t first, last; int rc; };
  std::deque<FailedRange> failed_ranges;
  std::vector<cudaEvent_t> timing_pool;
  std::chrono::steady_clock::time_point oldest_pending;
  uint64_t next_ticket = 0;
  uint64_t retired_through = 0;        /* every batch ticket up to here has finished and been retired */
  std::deque<Batch> batches;
  std::vector<cudaEvent_t> event_pool;
  TableSlot slots[kTableSlots];
  int next_slot = 0;

  uint32_t max_batch = 32, linger_us = 200;
  bool auto_register = false;          /* pin pageable host frames on first sight (opt-in) */
  /* automatic registrations by first byte: [lo, hi) and when it was last used. At most
   * auto_reg_limit () of them, least recently used dropped first. */
  struct AutoReg { uintptr_t hi; uint64_t tick; uintptr_t dev; /* device address of the first byte */ };
  std::map<uintptr_t, AutoReg> auto_regs;
  uint64_t auto_tick = 0;
  std::unordered_set<uint32_t> auto_streams;   /* streams whose frames have been registered */
  bool chroma_average = false;         /* fluc_ttmlblend_set_chroma_mode (1): NOT bit-exact */
  bool autocrop = true;                /* FLUC_TTMLBLEND_AUTOCROP=0: blend rectangles as handed in */
  bool use_groups = true;              /* FLUC_TTMLBLEND_GROUPS=0: generic table kernel only */
  bool eager_prepare = true;           /* FLUC_TTMLBLEND_EAGER_PREPARE=0: prepare at the first frame only */
  bool use_multi = true;               /* FLUC_TTMLBLEND_MULTI=0: dissolved groups go to the table kernel */
  bool profiling = false;
  uint32_t profile_every = 1, profile_seq = 0;   /* FLUC_TTMLBLEND_PROFILE_EVERY */
  /* FLUC_TTMLBLEND_SYNC=block: the events wait() / sync() sleep on are created with
   * cudaEventBlockingSync, so a waiting thread gives its core away instead of spinning (many
   * contexts / processes per box, tools/pcie_ceiling.cu); "spin" (default) has the lower latency */
  bool blocking_sync = false;
  std::thread sched;
  bool quit = false;

  /* staged host frames (staging.cu): FLUC_TTMLBLEND_STAGE_THREADS copy workers, at most
   * FLUC_TTMLBLEND_STAGE_SLOTS pinned staging frames in use */
  int stage_threads = 0, stage_slots_max = 64, stage_slots_total = 0;
  int stage_active = 0, stage_copying = 0;
  std::vector<PoolEntry> stage_slots_free;
  std::deque<std::shared_ptr<StageJob>> stage_in, stage_gpu, stage_out;
  std::map<uint64_t, std::shared_ptr<StageJob>> stage_jobs;      /* by blend_host ticket */
  std::condition_variable stage_cv, stage_gpu_cv, stage_done_cv;
  std::vector<std::thread> stage_workers;
  std::thread stage_completer;

  /* CPUs of the NUMA node the GPU hangs off (empty: unknown / disabled). Pinned host frames are
   * allocated with the calling thread moved there for the moment, so that their pages are local
   * to the GPU's PCIe root and zero-copy traffic does not cross the socket interconnect. */
  std::vector<int> numa_cpus;
  int numa_node = -1;
  std::vector<PoolEntry> pool_free, pool_used;
  /* pinned host frames are allocated several at a time, at a constant spacing: the frames a
   * pipeline takes from the pool one after the other then form runs that one two-dimensional
   * copy can move (host DMA batches, scheduler.cu) */
  std::vector<void *> host_slabs;
  /* host DMA batches (scheduler.cu). host_dma_policy: 0 never, 1 whenever a batch qualifies, 2 (default)
   * decided by measurement -- which of the two transports is faster depends on how the GPU hangs off
   * the host (measured: copy engines +12 % on a GPU with a root port of its own, -3.5 % on two GPUs
   * behind one bridge). DmaChoice: a trial of each transport over kDmaTrialFrames qualifying frames,
   * timed on the device between the completion of the trial's first and last batch, then the faster
   * one (zero copy unless the copy engines win by 2 %) for 2048, 8192, then kDmaSteadyFrames frames each time,
   * then again. */
  int host_dma_policy = 2;
  struct DmaChoice {
    int phase = 0;                     /* 0: trial of the copy engines, 1: trial of zero copy, 2: steady */
    bool dma = false;                  /* what the steady phase uses */
    int64_t left = 0;                  /* qualifying frames left in this phase (0: phase not begun) */
    cudaEvent_t ev[2][2] = { { nullptr, nullptr }, { nullptr, nullptr } };   /* [transport][begin, end], timing events */
    uint32_t frames[2] = { 0, 0 };     /* between begin and end */
    bool begun[2] = { false, false }, ended[2] = { false, false };
    bool judged = true;
    float rate[2] = { 0.f, 0.f };      /* frames per ms of the last trial */
    uint32_t trials = 0;
    bool cold = false;                 /* a staging set was allocated for this batch: not a batch to time */
    std::chrono::steady_clock::time_point last;   /* when the previous qualifying batch went out */
    uint32_t gaps = 0;                 /* trials given up because the caller paused in the middle */
  } dma_choice;
  bool dma_now () const {
    return host_dma_policy == 1 || (host_dma_policy == 2 && (dma_choice.phase == 0 || (dma_choice.phase == 2 && dma_choice.dma)));
  }
  uint32_t dma_piece = 8;              /* a batch for the copy engines goes out in pieces of this many frames, so that
                                        * the copy-out of one piece overlaps the copy-in of the next inside one call (0: whole) */
  cudaStream_t dma_in = nullptr, dma_out = nullptr;
  DmaSet dma_sets[kDmaSets];
  int next_dma_set = 0;
  uint32_t dma_outstanding = 0;        /* DMA batches in `batches` */
  std::vector<std::array<cudaEvent_t, 4>> dma_trace;   /* FLUC_TTMLBLEND_DMA_TRACE: copy-in begin / end, copy-out begin / end */
  std::unordered_set<const void *> pinned_planes;   /* plane pointers of the pinned host pool frames */
  uint8_t *scrub = nullptr;
  size_t scrub_bytes = 0;

  FlucTtmlBlendStats stats = {};
};

/* A failed allocation is reported and forgotten (the context stays usable); any other CUDA
 * error is sticky. */
#define CU(ctx, call) do {                                                   \
    cudaError_t e_ = (call);                                                 \
    if (e_ != cudaSuccess) {                                                 \
      (ctx)->cuda_error = std::string (#call) + ": " + cudaGetErrorString (e_); \
      if (e_ == cudaErrorMemoryAllocation) {                                 \
        cudaGetLastError ();                                                 \
        return FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY;                           \
      }                                                                      \
      (ctx)->sticky = FLUC_TTMLBLEND_ERROR_CUDA;                             \
      return FLUC_TTMLBLEND_ERROR_CUDA;                                      \
    }                                                                        \
  } while (0)

inline int
log_level ()
{
  static int lvl = -1;
  if (lvl < 0) {
    const char *e = getenv ("FLUC_TTMLBLEND_DEBUG");
    lvl = e ? atoi (e) : 0;
  }
  return lvl;
}

/* NVTX range for the current scope */
struct NvtxRange {
  explicit NvtxRange (const char *name) { nvtxRangePushA (name); }
  ~NvtxRange () { nvtxRangePop (); }
};

#define TBLOG(n, ...) do { if (log_level () >= (n)) { fprintf (stderr, "ttmlblend: " __VA_ARGS__); fputc ('\n', stderr); } } while (0)

/* overlay_cache.cu */
void free_deferred (Ctx *c, const std::vector<void *> &ptrs);
int prepare_overlay (Ctx *c, Overlay *ov, int format, int W, int H, Prepared **out);
std::vector<FlucTtmlBlendRect> disjoint_cover (const std::vector<FlucTtmlBlendRect> &in);
std::vector<int4> scale_row_plan (int src_h, int dst_h);
void crop_runs (const std::vector<int2> &spans, int min_gap, size_t max_runs, std::vector<FlucTtmlBlendRect> &out);
/* both are entered with the context lock held (lk), drop it while they upload, and return with
 * it held again whenever they got as far as dropping it */
int overlay_install (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, const FlucTtmlBlendRectangle *rects,
    uint32_t n, int image_w = 0, int image_h = 0);
int overlay_update_image (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, const uint8_t *bgra, int w, int h,
    int stride, const FlucTtmlBlendRect *changed, uint32_t n_changed);
int overlay_install_regions (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, int W, int H,
    const FlucTtmlBlendRegion *regions, uint32_t n);
/* ga: n values 0..255, one for every box or (n == 1) for all; mu held throughout */
int overlay_set_alpha (Ctx *c, uint32_t stream, const int *ga, uint32_t n);
/* x, y: one position per box (n == the number of rectangles installed); mu held throughout */
int overlay_set_positions (Ctx *c, uint32_t stream, const int32_t *x, const int32_t *y, uint32_t n);
/* render: one rectangle per box (n == the number of rectangles installed); entered with the
 * context lock held (lk), drops it while it waits for the scale and scan, returns with it held */
int overlay_set_render (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, const FlucTtmlBlendRect *render,
    uint32_t n);

/* jobs.cu */
void layout_spans (const Layout *L, std::vector<StageSpan> &out);
int check_frame (int fmt, int W, int H, const FlucTtmlBlendFrame *f);
uint64_t build_jobs (int format, int W, int H, uint32_t frame_flags, const FlucTtmlBlendFrame *src,
    const FlucTtmlBlendFrame *dst, const Prepared *prep, bool windowed, std::vector<PlaneJob> &jobs);
void make_groupable (Layout &L, bool lazy_inplace);
const Layout *find_layout (Ctx *c, Prepared *prep, bool lazy_inplace, int format, int W, int H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *src, const FlucTtmlBlendFrame *dst, bool windowed);
bool group_accepts (const Group &g, const PendingFrame &f);
void group_start (Group &g, const PendingFrame &f);
void group_add (Group &g, const PendingFrame &f);
void multi_start (MultiGroup &m, const PendingFrame &f);
bool multi_add (MultiGroup &m, const PendingFrame &f);
void emit_table_jobs (const std::vector<PlaneJob> &tmpl, const PendingFrame &f, std::vector<PlaneJob> *by_kind);

inline void
note_stream (Ctx *c, uint32_t stream)
{
  c->recent_streams[c->recent_pos] = stream;
  c->recent_pos = (c->recent_pos + 1) % 16;
  if (c->recent_n < 16)
    c->recent_n++;
}

inline bool
several_streams_active (const Ctx *c)
{
  for (uint32_t i = 1; i < c->recent_n; i++)
    if (c->recent_streams[i] != c->recent_streams[0])
      return true;
  return false;
}

/* fluc_ttmlblend.cu */
int queue_mapped_frame (Ctx *c, uint64_t tk, uint32_t stream, const std::shared_ptr<Overlay> &ov, Prepared *prep,
    int fmt, int W, int H, uint32_t frame_flags, const FlucTtmlBlendFrame *zf, const FlucTtmlBlendFrame *hf);

/* staging.cu */
int stage_frame (Ctx *c, std::unique_lock<std::mutex> &lk, uint64_t tk, uint32_t stream, const std::shared_ptr<Overlay> &ov,
    Prepared *prep, int fmt, int W, int H, uint32_t frame_flags, const FlucTtmlBlendFrame *hf);
int stage_wait (Ctx *c, std::unique_lock<std::mutex> &lk, uint64_t ticket, int *rc);
void stage_drain (Ctx *c, std::unique_lock<std::mutex> &lk, int phase);
void stage_shutdown (Ctx *c);
void stage_free_slots (Ctx *c);

/* scheduler.cu */
cudaEvent_t event_get (Ctx *c);
int launch_jobs (Ctx *c, TableSlot &s, const PlaneJob *jobs, size_t n, int kind, bool fast, int sync);
void reap_batches (Ctx *c);
int launch_pending (Ctx *c);
bool layout_takes_dma (const Layout *L);
void scheduler_main (Ctx *c);

}  // namespace tbh
#endif
