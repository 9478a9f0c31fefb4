/*
 * ttmlblend_kernels.cuh -- device-side data layout and launch interface of
 * the sm_100a blend / prepare kernels. Private to csrc/ (the public surface
 * is include/fluc_ttmlblend.h).
 *
 * Data layout in HBM (DESIGN.md "Data layout"):
 *   frames        planar / semi-planar / packed exactly as GStreamer maps them
 *                 (plane pointer + stride per plane).
 *   prepared      per overlay rectangle and per destination plane kind, the
 *   overlay       rectangle's pixels after everything that does not depend on
 *                 the frame has been done ONCE per cue change: BGRA unpack,
 *                 un-premultiply + BT.709 matrix (YUV destinations), global
 *                 alpha, 4:2:0 chroma siting (the even-x/even-y sample), and
 *                 shifting onto the 16-byte vector grid of the destination
 *                 plane. Two layouts:
 *                   PLANE8  alpha bytes + colour bytes, one of each per
 *                           destination byte (Y plane, U plane, V plane or
 *                           interleaved UV plane);
 *                   PACKED  one 32-bit word per pixel in the destination's
 *                           own channel order (AYUV / ARGB / ABGR: alpha in
 *                           byte 0, RGBA / BGRA: alpha in byte 3).
 */
#ifndef TTMLBLEND_KERNELS_CUH
#define TTMLBLEND_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>

namespace tb {

enum PlaneKind : int32_t {
  PK_PLANE8 = 0,
  PK_PACKED_A0 = 1,
  PK_PACKED_A3 = 2,
  PK_PLANE8_RGB = 3     /* 24-bit RGB / BGR: PLANE8's byte planes, RGB operators (premultiplied flag kept) */
};
constexpr int kPlaneKinds = 4;

enum JobFlags : int32_t {
  JF_VECTOR = 1,        /* src, dst and both pitches are 16-byte aligned */
  JF_INPLACE = 2,       /* dst == src: bytes no rectangle covers are not touched */
  JF_DST_PREMUL = 4,    /* destination frame is premultiplied (packed kinds) */
  JF_FAST = 8,          /* host-side: JF_VECTOR and no ragged last vector -> fast kernel */
  JF_LAZY = 16,         /* host-side, group launches in place: overlay first, skip transparent vectors */
  /* Programmatic dependent launch (set per launch, not part of a layout). Every blend launch of
   * the batch stream may start while its predecessor still runs -- frames of different batches
   * are independent unless the host's range tracker says otherwise:
   *   JF_PDL  launched with programmaticStreamSerializationAllowed: every CTA lets the next grid
   *           start at once (griddepcontrol.launch_dependents) and, when its own work is done,
   *           waits for the previous grid to have completed before it exits, so grids COMPLETE
   *           in launch order;
   *   JF_DEP  this launch touches memory an earlier launch that may still run reads or writes:
   *           its CTAs wait for the previous grid to complete (and with it every grid before
   *           that) before they touch anything. */
  JF_DEP = 32,
  JF_PDL = 64,
  JF_OPAQUE = 128,      /* host-side, group launches out of place: overlay first, no frame read under opaque vectors */
  JF_GA = 256           /* host-side, PLANE8 kinds: the launch holds a rectangle with RectRef::a_ga != 255 -> the
                         * variant that scales the prepared alpha bytes (overlay_set_global_alpha) */
};

/* One prepared rectangle as seen from one destination plane. */
struct alignas (16) RectRef {
  const uint8_t *a;     /* PLANE8: alpha bytes. PACKED: pixel words */
  const uint8_t *c;     /* PLANE8: colour bytes. PACKED: unused */
  int32_t v0, v1;       /* 16-byte vector columns [v0, v1) of the plane row */
  int32_t y0, y1;       /* plane rows [y0, y1); v0..y1 are read as one int4 */
  int32_t pitch;        /* bytes per prepared row, multiple of 16 */
  int32_t ga;           /* global alpha 0..255 of the Cs*ga terms (PACKED, PLANE8_RGB premultiplied) */
  int32_t src_premul;   /* PACKED: source colours are premultiplied */
  int32_t a_ga;         /* PLANE8 kinds: global alpha the blend still applies to the alpha bytes, asrc =
                         * a*a_ga/255 (JF_GA launches). 255 when it is 1 or the prepare folded it in */
};

enum JobClass : int32_t {
  JC_COPY = 0,          /* no rectangle touches the window */
  JC_ONE = 1,           /* one rectangle covers the whole window */
  JC_GENERAL = 2,       /* several rectangles and/or partial width */
  JC_ONE_BULK = 3       /* JC_ONE whose overlay bytes per chunk are contiguous (TMA staging) */
};

/* One window of one plane of one frame: a band of rows that all see the same
 * rectangles (rect_mask, bit i = rects[i]; every one of them spans all the
 * band's rows). Items are 16-byte vectors, numbered row-major inside the
 * window; a chunk is kItemsPerChunk consecutive items. */
struct alignas (16) PlaneJob {
  const uint8_t *src;
  uint8_t *dst;
  const RectRef *rects;
  unsigned long long rect_mask;
  int32_t src_pitch, dst_pitch;
  int32_t row_bytes;    /* valid bytes per plane row */
  int32_t win_v0, win_nv, win_y0, win_rows;
  uint32_t div_magic;   /* ceil (2^32 / win_nv): item / win_nv == umulhi (item, magic) */
  int32_t kind;         /* PlaneKind */
  int32_t flags;        /* JobFlags */
  int32_t cls;          /* JobClass */
  int32_t one_rect;     /* JC_ONE: index into rects */
  uint32_t n_chunks;
  int32_t plane;        /* host-side bookkeeping: plane index of the frame */
};

/* ---- group launch: frames that share geometry, tables in kernel parameters ---- */
constexpr int kMaxGroupFrames = 64;          /* multi-layout launches (parameter space) */
#ifndef TTMLBLEND_GROUP_FRAMES
#define TTMLBLEND_GROUP_FRAMES 256
#endif
constexpr int kMaxPlainGroupFrames = TTMLBLEND_GROUP_FRAMES;   /* plain group launches */
constexpr int kMaxGroupBands = 64;

struct BandDesc {             /* one band of rows of one plane, same for every frame */
  uint32_t chunk_begin;       /* first chunk of the band inside a frame's chunk list */
  int32_t plane;
  int32_t win_v0, win_nv, win_y0, win_rows;
  uint32_t div_magic;
  int32_t cls;                /* JobClass */
  int32_t one_rect;           /* JC_ONE: index into the plane's rectangle table */
  uint32_t rect_mask_lo, rect_mask_hi;
  uint32_t n_chunks;
};

struct FramePtrs {
  const uint8_t *src[3];
  uint8_t *dst[3];
  const RectRef *rects;       /* the frame's prepared overlay: all planes' tables, contiguous */
  uint64_t pad_;
};

struct GroupHeader {
  uint32_t n_frames, n_bands, chunks_per_frame, cpf_magic;
  uint32_t total_chunks, lanes, per_lane, lanes_magic;
  int32_t src_pitch[3], dst_pitch[3];
  int32_t rect_off[3];        /* first RectRef of plane p inside FramePtrs::rects */
  int32_t flags;              /* JobFlags shared by the group */
};

/* The parameter block of a group launch, sized by what it has to hold: a launch's parameters
 * are copied whole by the driver and fetched by the GPU's front end before the first CTA starts
 * (tools/launch_floor.cu: 3.0 us per launch with 1 KB of parameters, 5.1 us with 20 KB, 6.4 us
 * with 32 KB), which is most of the cost of a one-frame launch at 720p / 1080p. The host keeps
 * the full-size block and launches the smallest variant that fits. */
template <int NF, int NB>
struct GroupParamsT {
  GroupHeader h;
  BandDesc bands[NB];
  FramePtrs frames[NF];
};
using GroupParams = GroupParamsT<kMaxPlainGroupFrames, kMaxGroupBands>;           /* 19.5 KB */
using GroupParamsSmall = GroupParamsT<4, 16>;                                     /* 1.1 KB */
using GroupParamsMedium = GroupParamsT<32, kMaxGroupBands>;                       /* 5.2 KB */
/* > 4 KB of kernel parameters needs CUDA >= 12.1 and driver >= R530 (limit 32764 B), which
 * every sm_100a system has */
static_assert (sizeof (GroupParams) <= 32764, "kernel parameters");
static_assert (sizeof (GroupParamsSmall) <= 1280, "small group parameters");

/* ---- multi-layout group launch: frames of one format / size / pitch set whose cue layouts
 * (band lists) differ -- many streams, each showing its own text. Still everything in kernel
 * parameters: the distinct band lists back to back, and per frame its pointers, which band
 * list it uses and where its chunks start. */
constexpr int kMaxMultiBands = 576;

struct MultiParams {
  uint32_t n_frames, total_chunks, lanes, per_lane, lanes_magic;
  int32_t flags;
  int32_t src_pitch[3], dst_pitch[3];
  uint32_t frame_begin[kMaxGroupFrames + 1];      /* first chunk of every frame, then the total */
  uint16_t frame_band0[kMaxGroupFrames], frame_nbands[kMaxGroupFrames];
  FramePtrs frames[kMaxGroupFrames];              /* pad_ = rect_off of planes 0,1,2 in 16-bit fields */
  BandDesc bands[kMaxMultiBands];                 /* chunk_begin relative to the frame */
};
static_assert (sizeof (MultiParams) <= 32764, "kernel parameters");

constexpr int kThreads = 256;
#ifndef TTMLBLEND_UNROLL
#define TTMLBLEND_UNROLL 4
#endif
constexpr int kUnroll = TTMLBLEND_UNROLL;
constexpr int kItemsPerChunk = kThreads * kUnroll;

/* Parameters of the once-per-cue prepare kernels. Raw = device copy of the
 * rectangle's BGRA bytes whose pixel (0,0) sits at frame (fx, fy). */
struct PrepareParams {
  const uint8_t *raw;
  int32_t raw_pitch, raw_w, raw_h;
  int32_t fx, fy;
  int32_t cx0, cy0, cx1, cy1;   /* rectangle clipped to the frame */
  int32_t ga;                   /* (int) (255.0 * global_alpha) */
  int32_t premul;
  /* output */
  uint8_t *out_a, *out_c, *out_c2;
  int32_t out_pitch;
  int32_t v0;                   /* first vector column of the prepared span */
  int32_t row0, rows;           /* first plane row and number of prepared rows */
  int32_t mode;
  int32_t chroma_average;       /* non-parity option: 2x2 alpha-weighted chroma instead of the sited pixel */
  int32_t sub_x, sub_y;         /* chroma subsampling of the destination (2,2 / 2,1 / 1,1) */
};

enum PrepareMode : int32_t {
  PM_LUMA = 0,          /* out_a = alpha, out_c = Y, per pixel */
  PM_CHROMA_PLANAR = 1, /* out_a = alpha, out_c = U, out_c2 = V, per chroma sample */
  PM_CHROMA_UV = 2,     /* out_a = alpha pairs, out_c = U,V interleaved */
  PM_CHROMA_VU = 3,     /* out_a = alpha pairs, out_c = V,U interleaved */
  PM_PACKED_AYUV = 4,   /* words (A,Y,U,V) */
  PM_PACKED_ARGB = 5,
  PM_PACKED_ABGR = 6,
  PM_PACKED_RGBA = 7,
  PM_PACKED_BGRA = 8,
  PM_YUY2 = 9,          /* one plane, macropixels Y0 U Y1 V: out_a / out_c per byte */
  PM_UYVY = 10,         /* macropixels U Y0 V Y1 */
  PM_YVYU = 11,         /* macropixels Y0 V Y1 U */
  PM_VYUY = 12,         /* macropixels V Y0 U Y1 */
  PM_V308 = 13,         /* 3 bytes per pixel Y U V: out_a / out_c per byte, one thread per byte */
  PM_IYU2 = 14,         /* 3 bytes per pixel U Y V */
  PM_RGB24 = 15,        /* 3 bytes per pixel R G B, colour as in the source (no matrix) */
  PM_BGR24 = 16
};

/* One item of a batch prepare: one launch_prepare's work (n_elems elements per row, p.rows rows),
 * starting at CTA cta0 of the batch launch. */
struct alignas (16) PrepareItem {
  PrepareParams p;
  int32_t n_elems;
  uint32_t cta0;
};
/* items kept in the kernel parameters (4 KB of them); more are read from device memory */
constexpr uint32_t kPrepareBatchInline = 31;
struct PrepareBatch {
  const PrepareItem *items;     /* device copy of the items, or nullptr: inl */
  uint32_t n_items;
  uint32_t pad_[2];
  PrepareItem inl[kPrepareBatchInline];
};
static_assert (sizeof (PrepareBatch) <= 4096, "batch prepare parameters");

/* All jobs of one launch share one PlaneKind and one variant: fast (every
 * job 16-byte aligned with row_bytes % 16 == 0) or byte-granular. */
/* d_coarse[i] = index of the job that holds chunk i << kCoarseShift. */
constexpr int kCoarseShift = 4;
/* sync = JF_PDL / JF_DEP bits of this launch (0: an ordinary, fully serialised launch) */
/* ga: some job carries JF_GA (PLANE8 kinds): the variant that scales the prepared alpha bytes */
cudaError_t launch_blend (const PlaneJob *d_jobs, const uint32_t *d_chunk_begin, const uint32_t *d_coarse,
    int n_jobs, uint32_t total_chunks, int kind, bool fast, bool ga, int sync, cudaStream_t stream);
/* Fills in total_chunks and the interleave fields of P, then launches (the JF_GA variant when
 * P's flags carry it). */
cudaError_t launch_group (GroupParams &P, int kind, int sync, cudaStream_t stream);
/* Fills in total_chunks (from frame_begin[n_frames]) and the interleave fields, then launches. */
cudaError_t launch_multi (MultiParams &P, int kind, int sync, cudaStream_t stream);
/* n_elems = prepared elements per row (see PrepareMode). */
cudaError_t launch_prepare (const PrepareParams &p, int n_elems, cudaStream_t stream);
/* Fills in every item's cta0 (items without elements get none) and returns the CTAs of the batch. */
uint32_t prepare_batch_plan (PrepareItem *items, uint32_t n);
/* One launch of ttmlblend_prepare_batch_kernel for items[0..n) (n >= 1, planned): in the kernel
 * parameters when n <= kPrepareBatchInline, otherwise read from d_items, a device copy of them
 * ordered before the launch on `stream`. */
cudaError_t launch_prepare_batch (const PrepareItem *items, uint32_t n, const PrepareItem *d_items, uint32_t ctas,
    cudaStream_t stream);
cudaError_t launch_scrub (uint8_t *buf, size_t bytes, cudaStream_t stream);
/* bench helper: reads and rewrites `bytes` (multiple of 16) of mapped host memory in place */
cudaError_t launch_pcie_probe (uint8_t *buf, size_t bytes, cudaStream_t stream);
/* One TTML region composed onto the frame-sized premultiplied BGRA canvas (pixman 8-bit
 * arithmetic): background colour `bg` (premultiplied pixel, 0 = none), optional text layer,
 * group opacity mask `m8` (255 = none). Box already clipped to the canvas. */
struct RegionParams {
  uint8_t *canvas;
  int32_t canvas_pitch;
  int32_t x, y, w, h;           /* clipped box on the canvas */
  int32_t lx, ly;               /* canvas (x, y) is layer pixel (lx, ly) */
  const uint8_t *layer;         /* device copy or nullptr */
  int32_t layer_pitch;
  uint32_t bg;                  /* premultiplied a8r8g8b8 */
  uint32_t m8;
};
cudaError_t launch_region (const RegionParams &p, cudaStream_t stream);
/* (2r+1)^2 16.16 taps; ARGB32 in, ARGB32 out (pixman convolution semantics). */
cudaError_t launch_blur (const uint8_t *src, int w, int h, int src_pitch, const int32_t *taps, int radius,
    uint8_t *dst, int dst_pitch, cudaStream_t stream);
/* spans[y] = first / last x of row y with alpha != 0, (w, -1) for an empty row;
 * groups[y] = number of 16-pixel groups of the row with any alpha != 0. */
cudaError_t launch_rowspan (const uint8_t *raw, int pitch, int w, int h, int2 *spans, int *groups,
    cudaStream_t stream);
/* gst_video_blend_scale_linear_RGBA: rows[y] = (source row a, source row b, 8-bit weight, 0),
 * x_inc = the 16.16 horizontal increment; src needs dw's last position + 1 < its width. */
cudaError_t launch_scale (const uint8_t *src, int src_pitch, const int4 *rows, int x_inc, uint8_t *dst,
    int dst_pitch, int dw, int dh, cudaStream_t stream);

/* One rectangle of a resize (overlay_set_render_rectangles): scaled from its resident source to
 * w x h with the row plan at ScaleScanBatch::plans[plan ...] and x_inc as launch_scale, and its
 * rows scanned as launch_rowspan; plan < 0: the source is already w x h and is only scanned
 * (dst unused). Its rows are rows row0.. of the batch's spans / groups, and CTAs row0.. of the
 * launch. */
struct alignas (16) ScaleScanItem {
  const uint8_t *src;
  uint8_t *dst;
  int32_t src_pitch, dst_pitch;
  int32_t plan, x_inc;
  int32_t w, h;
  uint32_t row0;
  uint32_t pad_;
};
/* items kept in the kernel parameters; more are read from device memory */
constexpr uint32_t kScaleScanBatchInline = 32;
struct ScaleScanBatch {
  const ScaleScanItem *items;   /* device copy of the items, or nullptr: inl */
  const int4 *plans;            /* the row plans of every scaled item, back to back */
  int2 *spans;                  /* one per row of the batch; nullptr: no scan (no auto-crop) */
  int *groups;
  uint32_t n_items;
  uint32_t pad_[3];
  ScaleScanItem inl[kScaleScanBatchInline];
};
static_assert (sizeof (ScaleScanBatch) <= 4096, "scale-and-scan batch parameters");
/* Fills in every item's row0 and returns the rows (= CTAs) of the batch. */
uint32_t scale_scan_batch_plan (ScaleScanItem *items, uint32_t n);
/* One launch of ttmlblend_scale_scan_batch_kernel for items[0..n) (planned): in the kernel
 * parameters when n <= kScaleScanBatchInline, otherwise read from d_items, a device copy of them
 * ordered before the launch on `stream`. */
cudaError_t launch_scale_scan_batch (const ScaleScanItem *items, uint32_t n, const ScaleScanItem *d_items,
    const int4 *plans, int2 *spans, int *groups, uint32_t rows, cudaStream_t stream);

}  // namespace tb
#endif
