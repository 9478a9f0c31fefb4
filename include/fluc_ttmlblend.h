/*
 * fluc_ttmlblend.h -- C ABI of the B200 TTML overlay-blend path.
 *
 * One shared library, libfluc_ttmlblend.so, plain pointers and sizes, no GLib,
 * GStreamer, CUDA or torch types in any signature. Conventions follow the
 * reference's libs/fluc helpers (opaque `typedef struct _X X`, first argument
 * `thiz`, `fluc_<module>_<verb>`, FLUC_EXPORT, stats copied out under the
 * object's lock):
 *   /root/reference/libs/fluc/flu-codec-sdk/fluc/fluc_export.h:9-11
 *   /root/reference/libs/fluc/flu-codec-sdk/fluc/bwmeter/fluc_bwmeter.h:17-46
 *   /root/reference/libs/fluc/flu-codec-sdk/fluc/threads/fluc_monitor.h:15-44
 *
 * What it replaces. The reference's `ttmlrender` element produces one
 * premultiplied BGRA image per timeline interval
 * (/root/reference/plugins/ttml/gstttmlrender.c:1427-1478, caps :78-84) and
 * leaves the per-frame compositing to GStreamer (the README pipeline,
 * /root/reference/plugins/ttml/README.md:45-48), i.e. to gst-plugins-base:
 *   gboolean gst_video_overlay_composition_blend (GstVideoOverlayComposition *comp,
 *                                                 GstVideoFrame *video_buf);
 *   gboolean gst_video_blend (GstVideoFrame *dest, GstVideoFrame *src,
 *                             gint x, gint y, gfloat global_alpha);
 * The functions below take over exactly that work, bit for bit
 * (docs/BLENDSPEC.md), on the GPU. There is no CPU fallback: every entry point
 * returns FLUC_TTMLBLEND_ERROR_NO_DEVICE / _CUDA when the GPU cannot be used.
 *
 * Threading: every function may be called from any thread; a context
 * serialises internally (monitor = mutex + condition, fluc_monitor style).
 * `overlay_set*` is meant for the subtitle streaming thread (once per cue
 * change, the cadence of gst_ttmlbase_gen_buffer,
 * /root/reference/plugins/ttml/gstttmlbase.c:93-198), `submit*`/`blend_host`
 * for the video streaming threads of many elements at once.
 */
#ifndef _FLUC_TTMLBLEND_H_
#define _FLUC_TTMLBLEND_H_

#include <stddef.h>
#include <stdint.h>

#ifndef FLUC_EXPORT
#if defined(__GNUC__)
#define FLUC_EXPORT __attribute__ ((visibility ("default")))
#else
#define FLUC_EXPORT
#endif
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* One context per GPU: overlay cache, frame pool, batch scheduler, streams. */
typedef struct _FlucTtmlBlend FlucTtmlBlend;

/* Destination frame formats (GstVideoFormat names). */
typedef enum {
  FLUC_TTMLBLEND_FORMAT_I420 = 0,
  FLUC_TTMLBLEND_FORMAT_NV12 = 1,
  FLUC_TTMLBLEND_FORMAT_AYUV = 2,
  FLUC_TTMLBLEND_FORMAT_RGBA = 3,
  FLUC_TTMLBLEND_FORMAT_BGRA = 4,
  FLUC_TTMLBLEND_FORMAT_YV12 = 5,
  FLUC_TTMLBLEND_FORMAT_NV21 = 6,
  FLUC_TTMLBLEND_FORMAT_ARGB = 7,
  FLUC_TTMLBLEND_FORMAT_ABGR = 8,
  /* the padded RGB formats share pack/unpack with their alpha twins in GStreamer's format
   * table (PACK_RGBA / PACK_BGRA / PACK_ARGB / PACK_ABGR): the padding byte IS the alpha
   * byte as far as gst_video_blend is concerned, so these are the same code paths */
  FLUC_TTMLBLEND_FORMAT_RGBx = 9,
  FLUC_TTMLBLEND_FORMAT_BGRx = 10,
  FLUC_TTMLBLEND_FORMAT_xRGB = 11,
  FLUC_TTMLBLEND_FORMAT_xBGR = 12,
  /* further 8-bit YUV layouts GStreamer blends onto through the same AYUV lines: planar
   * 4:2:2 / 4:4:4, packed 4:2:2, grey. Chroma of a pixel pair comes from its even pixel. */
  FLUC_TTMLBLEND_FORMAT_Y42B = 13,
  FLUC_TTMLBLEND_FORMAT_Y444 = 14,
  FLUC_TTMLBLEND_FORMAT_YUY2 = 15,
  FLUC_TTMLBLEND_FORMAT_UYVY = 16,
  FLUC_TTMLBLEND_FORMAT_GRAY8 = 17,
  FLUC_TTMLBLEND_FORMAT_NV16 = 18,      /* semi-planar 4:2:2 */
  FLUC_TTMLBLEND_FORMAT_NV24 = 19,      /* semi-planar 4:4:4 */
  FLUC_TTMLBLEND_FORMAT_NV61 = 20,      /* NV16 with V before U */
  FLUC_TTMLBLEND_FORMAT_YVYU = 21,      /* packed 4:2:2, bytes Y0 V Y1 U */
  FLUC_TTMLBLEND_FORMAT_VYUY = 22,      /* packed 4:2:2, bytes V Y0 U Y1 */
  FLUC_TTMLBLEND_FORMAT_v308 = 23,      /* packed 4:4:4, 3 bytes per pixel: Y U V */
  FLUC_TTMLBLEND_FORMAT_IYU2 = 24,      /* packed 4:4:4, 3 bytes per pixel: U Y V */
  FLUC_TTMLBLEND_FORMAT_RGB = 25,       /* 24-bit R G B: no alpha byte, the destination counts as opaque */
  FLUC_TTMLBLEND_FORMAT_BGR = 26,
  FLUC_TTMLBLEND_FORMAT_COUNT
} FlucTtmlBlendFormat;

/* Error codes: 0 = ok, negative = error. Never aborts. */
typedef enum {
  FLUC_TTMLBLEND_OK = 0,
  FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT = -1,
  FLUC_TTMLBLEND_ERROR_NO_DEVICE = -2,     /* no usable CUDA device */
  FLUC_TTMLBLEND_ERROR_CUDA = -3,          /* sticky: context is unusable */
  FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY = -4,  /* this call failed; the context stays usable */
  FLUC_TTMLBLEND_ERROR_UNSUPPORTED_FORMAT = -5,
  FLUC_TTMLBLEND_ERROR_NOT_FOUND = -6,     /* unknown stream / ticket / frame */
  FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES = -7
} FlucTtmlBlendError;

/* Mirrors GST_VIDEO_OVERLAY_FORMAT_FLAG_PREMULTIPLIED_ALPHA (rectangles) and
 * GST_VIDEO_FLAG_PREMULTIPLIED_ALPHA (frames). */
#define FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA 1u

#define FLUC_TTMLBLEND_MAX_RECTANGLES 64u

/* A region of the frame, in frame pixels; may extend beyond the frame.
 * Source of these in the reference: GstTTMLRegion origin/extent,
 * /root/reference/plugins/ttml/gstttmlrender.c:44-76,434-561. */
typedef struct {
  int32_t x, y, w, h;
} FlucTtmlBlendRect;

/* One overlay rectangle = GstVideoOverlayRectangle: BGRA bytes (ARGB32 little
 * endian), position, global alpha, premultiplied flag, render size. ttmlrender's
 * image is rendered at its pixel size (render_width = render_height = 0); a
 * rectangle with another render size is first scaled on the GPU exactly as
 * gst_video_overlay_composition_blend does with gst_video_blend_scale_linear_RGBA
 * (once per cue, cached like everything else); its pixel size must then be >= 2x2,
 * and neither its pixel size nor its render size may exceed 32768 on either side
 * (the scaler's 16.16 positions are 32-bit): FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT
 * otherwise. render_width / render_height above 32768 are refused in any case. */
typedef struct {
  const uint8_t *pixels;   /* host memory -- or device memory of the context's GPU: a cue that is
                            * already in HBM is copied there -- read before the call returns */
  int32_t width, height, stride;
  int32_t x, y;
  float global_alpha;      /* 1.0f for ttmlrender */
  uint32_t flags;          /* FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA */
  int32_t render_width, render_height;   /* 0 = width / height (no scaling) */
} FlucTtmlBlendRectangle;

/* Plane pointers + strides of one frame (GstVideoFrame data[]/stride[]).
 * I420 / Y42B / Y444: Y,U,V. YV12: Y,V,U. NV12/NV21/NV16/NV61/NV24: Y,UV. Packed formats, GRAY8: plane[0]. */
typedef struct {
  void *plane[3];
  int32_t stride[3];
} FlucTtmlBlendFrame;

/* Counters, copied out like fluc_bwmeter_stats_copy
 * (/root/reference/libs/fluc/flu-codec-sdk/fluc/bwmeter/fluc_bwmeter.c:71-76). */
typedef struct {
  uint64_t frames_blended;      /* frames that went through a blend launch */
  uint64_t launches;            /* blend kernel launches */
  uint64_t group_launches;      /* of which: group launches (tables in kernel parameters) */
  uint64_t prepare_launches;    /* overlay prepare kernel launches */
  uint64_t overlays_set;
  uint64_t algorithmic_bytes;   /* 2*frame bytes (or touched bytes in place) + 4*overlay px */
  uint64_t h2d_bytes, d2h_bytes;   /* zero-copy host frames: bytes of the windows under the cue (an
                                    * upper bound when a lazy launch skips transparent vectors or
                                    * does not read under opaque ones) */
  double kernel_ms;             /* sum of the CUDA-event times of the timed batches (profiling on) */
  uint64_t kernel_ms_launches;  /* batches included in kernel_ms (one launch each unless mixed) */
  uint64_t cache_bytes;         /* device memory held by overlay caches right now (stream-ordered pool) */
  uint64_t multi_launches;      /* launches that carried frames with different cue layouts (band
                                 * lists of up to 64 frames in the kernel parameters) */
  uint64_t lazy_launches;       /* launches in place that read the overlay first: vectors it leaves
                                 * untouched are skipped, vectors it covers opaquely are written
                                 * without being read (sparse cues, opaque boxes; exact either way) */
  uint64_t host_dma_batches;    /* batches of pinned host frames moved by the copy engines (2-D copies of
                                 * the rows under the cue, frames at a constant spacing) instead of
                                 * being read and written by the kernel over PCIe */
  uint64_t opaque_skip_launches; /* launches out of place that read the overlay first and do not read the
                                 * frame under vectors it covers opaquely (cues with an opaque box) */
  uint64_t staged_frames;       /* host frames the GPU could not reach directly (pageable or unaligned
                                 * memory): their cue rows went through pinned staging frames */
  uint64_t overlays_updated;    /* of overlays_set: cue changes that kept the untouched regions (overlay_update) */
  uint64_t dependent_launches;  /* batches that had to wait for everything launched before them: they
                                 * write what an earlier batch that may still run reads or writes, or
                                 * read what it writes (all others may overlap their predecessor's tail:
                                 * programmatic dependent launch) */
} FlucTtmlBlendStats;

/* ---- lifetime -------------------------------------------------------- */
FLUC_EXPORT int fluc_ttmlblend_new (int device, FlucTtmlBlend **out);
FLUC_EXPORT void fluc_ttmlblend_free (FlucTtmlBlend *thiz);
FLUC_EXPORT const char *fluc_ttmlblend_strerror (int err);
/* Text of the last CUDA error seen by this context ("" if none). */
FLUC_EXPORT const char *fluc_ttmlblend_last_cuda_error (FlucTtmlBlend *thiz);
FLUC_EXPORT int fluc_ttmlblend_device_count (void);
/* NUMA node of the context's GPU (-1: unknown or FLUC_TTMLBLEND_NUMA=0). Pinned pool frames
 * (frame_pool_acquire with on_host) are allocated on that node. */
FLUC_EXPORT int fluc_ttmlblend_numa_node (FlucTtmlBlend *thiz);
FLUC_EXPORT const char *fluc_ttmlblend_version (void);

/* ---- several GPUs in one process --------------------------------------
 * Streams are independent, so a process that serves many of them (one GStreamer process,
 * many elements) spreads them over the box's GPUs with no exchange between GPUs: one
 * context per device, stream s lives on context s % n (SURVEY.md section 8e; the same
 * partition flu-plugins-oss_b200/sharding.py uses across processes). Everything about a
 * stream -- overlay_set, submit, blend_host, wait, pool frames -- is then done on
 * fluc_ttmlblend_multi_context (m, stream). */
typedef struct _FlucTtmlBlendMulti FlucTtmlBlendMulti;
/* devices == NULL or n_devices == 0: every CUDA device of the box. */
FLUC_EXPORT int fluc_ttmlblend_multi_new (const int *devices, uint32_t n_devices, FlucTtmlBlendMulti **out);
FLUC_EXPORT void fluc_ttmlblend_multi_free (FlucTtmlBlendMulti *thiz);
FLUC_EXPORT uint32_t fluc_ttmlblend_multi_size (FlucTtmlBlendMulti *thiz);
FLUC_EXPORT FlucTtmlBlend *fluc_ttmlblend_multi_context (FlucTtmlBlendMulti *thiz, uint32_t stream);
FLUC_EXPORT int fluc_ttmlblend_multi_device (FlucTtmlBlendMulti *thiz, uint32_t stream);
FLUC_EXPORT int fluc_ttmlblend_multi_sync (FlucTtmlBlendMulti *thiz);     /* flush + wait, every device */

/* ---- overlay cache: once per cue change ------------------------------ */
/* ttmlrender form: one W*H premultiplied BGRA image (gen_buffer output) plus
 * the region rectangles that can hold non-transparent pixels. n_rects == 0
 * means the whole image is one rectangle. Replaces the stream's previous
 * overlay atomically; frames already submitted keep the old one. */
FLUC_EXPORT int fluc_ttmlblend_overlay_set (FlucTtmlBlend *thiz, uint32_t stream,
    const uint8_t *bgra_premul, int32_t w, int32_t h, int32_t stride,
    const FlucTtmlBlendRect *rects, uint32_t n_rects);
/* The next state of the same cue: ttmlrender re-renders its whole image for every timeline
 * event, including <set> animation steps and roll-up lines
 * (/root/reference/plugins/ttml/gstttmlrender.c:1442-1452,
 * /root/reference/plugins/ttml/gstttmlevent.c:208-233, /root/reference/plugins/ttml/gstttmlstyle.c:286-312),
 * while only some regions differ from the image before. `bgra_premul` is the new w*h image,
 * `changed_rects` cover every pixel that differs from the image the stream's overlay was built
 * from (by overlay_set or a previous overlay_update, same w and h). Region boxes the changed
 * rectangles do not touch keep their device pixels, their crop and their prepared planes; only
 * the touched boxes are uploaded and prepared again. The result is the same as overlay_set with
 * the new image and the old region boxes, swapped in as atomically. Falls back to installing the
 * whole image (overlay_set without boxes) when the stream has no such overlay or a change lies
 * outside every region box. n_changed == 0: nothing changed, nothing is done. */
FLUC_EXPORT int fluc_ttmlblend_overlay_update (FlucTtmlBlend *thiz, uint32_t stream,
    const uint8_t *bgra_premul, int32_t w, int32_t h, int32_t stride,
    const FlucTtmlBlendRect *changed_rects, uint32_t n_changed);
/* GstVideoOverlayComposition form: independent rectangles, blended in order. Each rectangle is
 * kept whole on the device, also the part that lies above or left of the frame (or all of it),
 * so that overlay_set_positions can move it in later: such rectangles count those pixels in
 * h2d_bytes and cache_bytes. A rectangle with another render size also keeps its pixels at their
 * own size, so that overlay_set_render_rectangles can scale it again: cache_bytes counts them
 * besides the scaled image. The blended frames do not depend on it. */
FLUC_EXPORT int fluc_ttmlblend_overlay_set_rectangles (FlucTtmlBlend *thiz,
    uint32_t stream, const FlucTtmlBlendRectangle *rects, uint32_t n_rects);
/* Region form (SURVEY.md section 8f rank 3): the overlay is composed on the GPU from region
 * descriptors instead of being drawn by Cairo on the host -- what
 * gst_ttmlrender_show_regions does around the text
 * (/root/reference/plugins/ttml/gstttmlrender.c:1250-1268,1375-1381): background fill,
 * group opacity, regions in list (z-index) order. `layer`, if not NULL, is what the host
 * rasterised for the region's text/outline on a CLEARED w*h surface (premultiplied BGRA);
 * it is composited OVER the background. Arithmetic: Cairo's colour conversion and
 * pixman's 8-bit premultiplied OVER / IN (docs/BLENDSPEC.md section 9); parity with a real
 * Cairo is unpinned, and a layer is only equivalent to Cairo drawing the glyphs one by one
 * where anti-aliased glyph edges do not overlap. */
typedef struct {
  int32_t x, y, w, h;            /* GstTTMLRegion originx/y, extentx/y (gstttmlrender.c:44-76) */
  uint32_t background_color;     /* 0xRRGGBBAA (gstttmlattribute.c:22); 0 = none */
  double opacity;                /* tts:opacity, 1.0 = none */
  const uint8_t *layer;          /* optional, host memory, read before the call returns */
  int32_t layer_stride;
} FlucTtmlBlendRegion;
FLUC_EXPORT int fluc_ttmlblend_overlay_set_regions (FlucTtmlBlend *thiz, uint32_t stream,
    int32_t frame_width, int32_t frame_height, const FlucTtmlBlendRegion *regions, uint32_t n_regions);
/* The "clear" buffer ttmlrender pushes for timeline gaps
 * (/root/reference/plugins/ttml/gstttmlevent.c:221-224): frames pass through. */
FLUC_EXPORT int fluc_ttmlblend_overlay_clear (FlucTtmlBlend *thiz, uint32_t stream);

/* gst_video_overlay_rectangle_set_global_alpha for the stream's current overlay, without a new
 * upload or prepare: a fade costs a few hundred bytes of rectangle tables instead of a cue change.
 * n == 1: every rectangle gets global_alpha[0]. Otherwise n == the number of rectangles the
 * overlay was installed with, one value each: overlay_set_rectangles: the list, in order (also
 * rectangles that lie outside the frame); overlay_set: its region boxes as installed, i.e.
 * clipped to the image, overlapping boxes split into disjoint ones (1 without boxes);
 * overlay_set_regions: 1, its regions are composed into one image first. Values in [0, 1].
 * Replaces the values, as set_global_alpha does. Frames submitted after the call (submit*,
 * submit_many_after, blend_host*) are blended exactly as gst_video_blend does with those global
 * alphas (ga = (int) (255.0 * global_alpha)); frames already submitted keep theirs.
 * overlay_update keeps the current values when it patches the overlay (when it falls back to
 * installing the whole image, that starts at 1); overlay_set* / overlay_clear start again from
 * the new cue's own values. A rectangle installed with a global alpha below 1 is prepared once
 * more the first time its value changes.
 * Returns NOT_FOUND when the stream has no overlay, INVALID_ARGUMENT for a wrong n, NULL, NaN or
 * a value outside [0, 1]. */
FLUC_EXPORT int fluc_ttmlblend_overlay_set_global_alpha (FlucTtmlBlend *thiz, uint32_t stream,
    const float *global_alpha, uint32_t n);

/* gst_video_overlay_rectangle_set_render_rectangle for the position only: rectangle i of the
 * stream's overlay_set_rectangles list (in list order, including rectangles outside the frame)
 * is placed at (x[i], y[i]). Nothing is uploaded, scaled or scanned again. The render size stays
 * the one the rectangle was installed with (overlay_set_render_rectangles changes it). Frames submitted after the call (submit*,
 * submit_many_after, blend_host*) are blended exactly as overlay_set_rectangles with the moved
 * rectangles would blend them. Frames already submitted keep the old positions.
 * The rectangles keep their current global alphas, and overlay_set_global_alpha after a move
 * keeps the positions; overlay_set* / overlay_clear start again from the new cue. A move
 * prepares the moved rectangles again from their resident pixels on the GPU, in one kernel
 * launch per destination format and size the stream has been blended in (under
 * FLUC_TTMLBLEND_CHROMA_AVERAGE, plus one launch per moved rectangle for its averaged chroma).
 * Unchanged positions: nothing is done. Returns NOT_FOUND when the stream has no overlay,
 * INVALID_ARGUMENT for NULL arrays, n different from the number of rectangles installed, an
 * overlay installed by overlay_set, overlay_update or overlay_set_regions, or a position at which
 * x + render width or y + render height overflows int32_t. */
FLUC_EXPORT int fluc_ttmlblend_overlay_set_positions (FlucTtmlBlend *thiz, uint32_t stream,
    const int32_t *x, const int32_t *y, uint32_t n);

/* gst_video_overlay_rectangle_set_render_rectangle, position and size: rectangle i of the
 * stream's overlay_set_rectangles list (in list order, as for overlay_set_positions) is placed at
 * (render[i].x, render[i].y) and rendered at render[i].w x render[i].h; a side of 0 means the pixel
 * size, as render_width = 0 does at install. Nothing is uploaded: a rectangle whose size changes is
 * scaled again on the GPU from the pixels it was installed with, exactly as overlay_set_rectangles
 * scales (or, back at its pixel size, taken as it is), and cropped again to its non-transparent
 * rows. Frames submitted after the call (submit*, submit_many_after, blend_host*) are blended
 * exactly as overlay_set_rectangles with the same pixels, flags and current global alphas at the
 * new render rectangles would blend them. Frames already submitted keep the old geometry.
 * The rectangles keep their current global alphas; overlay_set_global_alpha and
 * overlay_set_positions after a resize keep the new sizes. Cost: every resized rectangle is scaled
 * and scanned in one kernel launch whose row spans the call waits for (one host wait per call),
 * then prepared as a move prepares (one launch per destination format and size the stream has been
 * blended in; under FLUC_TTMLBLEND_CHROMA_AVERAGE, plus one per resized rectangle). An entry whose
 * size stays and whose position changes costs what overlay_set_positions costs; nothing changed:
 * nothing is done. Returns NOT_FOUND when the stream has no overlay (or another thread replaced it
 * while the call waited), INVALID_ARGUMENT for a NULL array, n different from the number of
 * rectangles installed, an overlay installed by overlay_set, overlay_update or
 * overlay_set_regions, a side below 0 or above 32768, a rectangle that would be scaled while its
 * pixel size is below 2x2 or above 32768 on a side, or x + w or y + h overflowing int32_t. A
 * refused call changes nothing. */
FLUC_EXPORT int fluc_ttmlblend_overlay_set_render_rectangles (FlucTtmlBlend *thiz, uint32_t stream,
    const FlucTtmlBlendRect *render, uint32_t n);

/* How the overlay reaches the chroma planes of 4:2:0 frames. SITED (default) is what
 * GStreamer does and the only bit-exact mode: a chroma sample takes the overlay pixel at
 * (even x, even y). AVERAGE is an explicit NON-PARITY option: the alpha-weighted mean of
 * the 2x2 pixels (no chroma fringes under anti-aliased glyph edges). Applies to overlays
 * prepared after the call. */
#define FLUC_TTMLBLEND_CHROMA_SITED 0
#define FLUC_TTMLBLEND_CHROMA_AVERAGE 1
FLUC_EXPORT int fluc_ttmlblend_set_chroma_mode (FlucTtmlBlend *thiz, int mode);

/* ---- per frame, device-resident (batched) ---------------------------- */
/* Queues one frame. src/dst hold DEVICE pointers; dst == src (same plane[0])
 * blends in place like gst_video_blend does, otherwise the whole frame is
 * written to dst. frame_flags: FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA for a
 * premultiplied destination. The batch is launched by flush(), by wait() on
 * one of its tickets, when it reaches the batch limit, or by the scheduler
 * thread after the linger time. */
FLUC_EXPORT int fluc_ttmlblend_submit (FlucTtmlBlend *thiz, uint32_t stream,
    FlucTtmlBlendFormat fmt, int32_t width, int32_t height, uint32_t frame_flags,
    const FlucTtmlBlendFrame *src, const FlucTtmlBlendFrame *dst,
    uint64_t *ticket);
/* The same for n frames of one geometry under a single lock (many streams, or
 * consecutive frames of one): streams[i], srcs[i], dsts[i], tickets[i]. */
FLUC_EXPORT int fluc_ttmlblend_submit_many (FlucTtmlBlend *thiz, uint32_t n,
    const uint32_t *streams, FlucTtmlBlendFormat fmt, int32_t width, int32_t height,
    uint32_t frame_flags, const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts,
    uint64_t *tickets);
FLUC_EXPORT int fluc_ttmlblend_flush (FlucTtmlBlend *thiz);
/* Returns when the frame is complete. A frame that is still queued is launched at once when its
 * stream is the only active one; when several streams have been submitting, the batch is left
 * to the scheduler thread for up to the linger time (or until it is full) so that synchronous
 * callers of different streams share launches. linger_us = 0 turns that off. */
FLUC_EXPORT int fluc_ttmlblend_wait (FlucTtmlBlend *thiz, uint64_t ticket);
/* flush + wait for everything in flight at the time of the call (the context is not locked
 * while waiting: other threads keep submitting). */
FLUC_EXPORT int fluc_ttmlblend_sync (FlucTtmlBlend *thiz);
/* Scheduler knobs: frames per launch (default 32, 1..1024) and how long the
 * scheduler thread lets a partial batch linger, in microseconds (default 200;
 * 0 = no scheduler thread launches, only flush/wait/limit). */
FLUC_EXPORT int fluc_ttmlblend_set_batch (FlucTtmlBlend *thiz, uint32_t max_frames,
    uint32_t linger_us);

/* ---- per frame, device-resident, ordered by the caller's CUDA stream --
 * For frames another CUDA stream produces and consumes (decoder -> blend -> encoder), without a
 * host thread blocking in between. `cuda_stream` is a cudaStream_t of the context's device passed
 * as a pointer; NULL is the legacy default stream of that device. A stream of another device is
 * INVALID_ARGUMENT.
 *
 * submit_many_after: submit_many, ordered after everything enqueued on cuda_stream before this
 * call: the frames' launch does not start reading or writing them until that work is complete.
 * The host never waits for it, with one exception: table-kernel launches rotate through 8 job-table
 * slots, and a ninth such launch while 8 are held back waits for the first. The call records one
 * event on cuda_stream; the launch that carries the call's frames waits for it on the blend stream
 * (not at all when it has already completed). Such a launch goes out as an ordinary launch, not a
 * programmatic dependent one. Frames of different calls, and submit* frames, still share launches:
 * such a launch waits for all of its producers.
 *
 * wait_on_stream: work enqueued on cuda_stream after this call runs after the ticket's frame is
 * complete. The ticket resolves as in wait(): NOT_FOUND for 0 or a ticket not handed out yet,
 * nothing enqueued for a frame already complete, the error of a launch that failed. A frame that
 * is still queued is launched under the same policy as wait() (it may linger for up to the linger
 * time while several streams are active). The host never waits for the GPU. A host frame that
 * went through the staging threads (blend_host of memory the GPU cannot reach) ends with a CPU
 * copy no stream can wait for: INVALID_ARGUMENT, use wait(). Zero-copy host frames are fine.
 *
 * Batches complete in launch order, so waiting for the last ticket of a call covers every frame
 * of it, even when the batch limit or a dependency between its frames split it into several
 * launches.
 *
 * A frame may be reused -- rewritten by its producer, or freed -- only after its ticket has been
 * waited for: with wait(), or with wait_on_stream() on the stream that reuses it. */
FLUC_EXPORT int fluc_ttmlblend_submit_many_after (FlucTtmlBlend *thiz, void *cuda_stream,
    uint32_t n, const uint32_t *streams, FlucTtmlBlendFormat fmt, int32_t width, int32_t height,
    uint32_t frame_flags, const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts,
    uint64_t *tickets);
FLUC_EXPORT int fluc_ttmlblend_wait_on_stream (FlucTtmlBlend *thiz, uint64_t ticket, void *cuda_stream);

/* ---- per frame, host-resident: the drop-in for -----------------------
 * gst_video_overlay_composition_blend (comp, frame). The frame is in HOST
 * memory and is modified in place; only the rows (and columns) the cue covers
 * cross PCIe. Device-accessible frames -- pool frames acquired with on_host=1,
 * or memory passed to host_register, 16-byte aligned -- are blended zero copy:
 * they join the batch like submit() frames and the kernel reads and writes
 * them over PCIe itself. Anything else (pageable or unaligned memory) is
 * staged by worker threads: the rows under the cue are copied into a pinned
 * staging frame, blended zero copy, and copied back.
 * Asynchronous either way: the frame is complete once wait(ticket) returns. */
FLUC_EXPORT int fluc_ttmlblend_blend_host (FlucTtmlBlend *thiz, uint32_t stream,
    FlucTtmlBlendFormat fmt, int32_t width, int32_t height, uint32_t frame_flags,
    const FlucTtmlBlendFrame *host_frame, uint64_t *ticket);
/* The same for n host frames of one geometry under a single lock (many streams, or a run of
 * frames of one): streams[i], host_frames[i], tickets[i]. Waiting for the last ticket waits
 * for all of them when every frame took the zero-copy path. */
FLUC_EXPORT int fluc_ttmlblend_blend_host_many (FlucTtmlBlend *thiz, uint32_t n,
    const uint32_t *streams, FlucTtmlBlendFormat fmt, int32_t width, int32_t height,
    uint32_t frame_flags, const FlucTtmlBlendFrame *host_frames, uint64_t *tickets);
/* Opt-in: pin pageable host frames the first time blend_host sees them (48 planes per stream
 * that uses it, at least 192; least recently used dropped), so that recycled buffers of a pool
 * take the zero-copy path. A registration pins the physical pages: whoever owns such memory MUST
 * call host_forget (or host_unregister) before freeing it -- a later allocation at the same
 * address would otherwise be taken for the registered one while the GPU still reaches the old
 * pages. (The GStreamer glue does so from the GstMemory's destroy notification.) */
FLUC_EXPORT int fluc_ttmlblend_set_auto_register (FlucTtmlBlend *thiz, int enabled);
/* How batches of pinned pool frames (fluc_ttmlblend_frame_acquire with on_host=1, which come in
 * slabs of constant spacing) cross PCIe. mode 0: zero copy only -- the kernel reads the rows under
 * the cue from host memory and writes them back. mode 1: the copy engines whenever a batch
 * qualifies (at least 4 in-place frames of one layout with full-row translucent windows) -- two-
 * dimensional copies of the rows under the cue for a whole run of frames, 8 frames at a time, blended
 * in device staging and copied back on a third stream. mode 2 (the default; FLUC_TTMLBLEND_HOST_DMA
 * presets the mode): measured -- a trial of either transport over 128 qualifying frames, timed on the
 * device, then the faster one for 32768 frames, then again. Which one wins depends on how the GPU
 * hangs off the host: +12 % for the copy engines on a GPU with a root port of its own (14.8 k against
 * 13.2 k frames/s, 4K NV12), -3.5 % on two GPUs behind one host bridge. Results are identical
 * either way. */
FLUC_EXPORT int fluc_ttmlblend_set_host_dma (FlucTtmlBlend *thiz, int mode);
FLUC_EXPORT int fluc_ttmlblend_host_register (FlucTtmlBlend *thiz, void *ptr, size_t bytes);
/* Both wait for every frame of the context that is queued or in flight before they unpin. */
FLUC_EXPORT int fluc_ttmlblend_host_unregister (FlucTtmlBlend *thiz, void *ptr);
/* Drops every AUTOMATIC registration that intersects [ptr, ptr + bytes). Returns how many
 * there were (>= 0), or a negative error. Memory that was never seen is not an error. */
FLUC_EXPORT int fluc_ttmlblend_host_forget (FlucTtmlBlend *thiz, const void *ptr, size_t bytes);

/* ---- frame pool ------------------------------------------------------ */
/* Device frames (HBM) or pinned host staging frames, recycled by geometry.
 * Planes are 256-byte aligned with a 256-byte multiple stride. */
FLUC_EXPORT int fluc_ttmlblend_frame_pool_acquire (FlucTtmlBlend *thiz,
    FlucTtmlBlendFormat fmt, int32_t width, int32_t height, int on_host,
    FlucTtmlBlendFrame *out);
FLUC_EXPORT int fluc_ttmlblend_frame_pool_release (FlucTtmlBlend *thiz,
    const FlucTtmlBlendFrame *frame);
/* Synchronous whole-frame copies between a host frame and a device frame. */
FLUC_EXPORT int fluc_ttmlblend_frame_upload (FlucTtmlBlend *thiz,
    FlucTtmlBlendFormat fmt, int32_t width, int32_t height,
    const FlucTtmlBlendFrame *host_src, const FlucTtmlBlendFrame *dev_dst);
FLUC_EXPORT int fluc_ttmlblend_frame_download (FlucTtmlBlend *thiz,
    FlucTtmlBlendFormat fmt, int32_t width, int32_t height,
    const FlucTtmlBlendFrame *dev_src, const FlucTtmlBlendFrame *host_dst);
/* Plane geometry of a format (rows and valid bytes per row). */
FLUC_EXPORT int fluc_ttmlblend_format_planes (FlucTtmlBlendFormat fmt);
FLUC_EXPORT int fluc_ttmlblend_plane_row_bytes (FlucTtmlBlendFormat fmt, int plane, int32_t width);
FLUC_EXPORT int fluc_ttmlblend_plane_rows (FlucTtmlBlendFormat fmt, int plane, int32_t height);

/* ---- producer-side helper: textOutline blur (once per cue) ----------- */
/* gst_ttml_blur_image_surface (surface, radius, sigma) of
 * /root/reference/plugins/ttml/gstttmlblur.c:72-110 on the GPU: Gaussian
 * kernel of (2*radius+1)^2 16.16 fixed-point taps, pixman convolution
 * semantics (transparent outside the image, (sum + 0x8000) >> 16, clip).
 * ARGB32 in host memory in, ARGB32 out; synchronous. radius 0..64. */
FLUC_EXPORT int fluc_ttmlblend_blur_argb32 (FlucTtmlBlend *thiz, const uint8_t *src,
    int32_t width, int32_t height, int32_t stride, int32_t radius, double sigma,
    uint8_t *dst, int32_t dst_stride);

/* ---- observability --------------------------------------------------- */
FLUC_EXPORT void fluc_ttmlblend_stats_copy (FlucTtmlBlend *thiz, FlucTtmlBlendStats *out);
FLUC_EXPORT void fluc_ttmlblend_stats_reset (FlucTtmlBlend *thiz);
/* Sum over the contexts of a multi (kernel_ms adds up device time spent in parallel). */
FLUC_EXPORT void fluc_ttmlblend_multi_stats_copy (FlucTtmlBlendMulti *thiz, FlucTtmlBlendStats *out);
/* Per-launch CUDA-event timing of the blend kernel into stats.kernel_ms:
 * 0 = off, 1 = every launch, n > 1 = every n-th launch (an event pair between
 * two launches keeps them from overlapping, ~2 % at 4K x 32 frames). */
FLUC_EXPORT int fluc_ttmlblend_set_profiling (FlucTtmlBlend *thiz, int enabled);
/* Device timer on the blend stream: begin records an event, end records a
 * second one, waits for it and returns the milliseconds in between. */
FLUC_EXPORT int fluc_ttmlblend_timer_begin (FlucTtmlBlend *thiz);
FLUC_EXPORT int fluc_ttmlblend_timer_end (FlucTtmlBlend *thiz, double *ms);
/* Writes `bytes` of device memory on the blend stream (L2 flush for benches). */
FLUC_EXPORT int fluc_ttmlblend_scrub_l2 (FlucTtmlBlend *thiz, size_t bytes);
/* Bench helper: `repeats` x submit_many of the same n frames (plus a flush each time the batch
 * limit did not launch it) without returning to the caller in between. For one-frame batches a
 * scripting-language loop around submit_many costs several times the launch itself. dsts holds
 * dst_sets x n frames; repeat r writes into set r % dst_sets, as the frames of a running
 * pipeline come out of a buffer pool rather than landing in the same buffers every time. */
FLUC_EXPORT int fluc_ttmlblend_submit_many_repeat (FlucTtmlBlend *thiz, uint32_t n,
    const uint32_t *streams, FlucTtmlBlendFormat fmt, int32_t width, int32_t height,
    uint32_t frame_flags, const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts,
    uint32_t dst_sets, uint32_t repeats);
/* Bench helper: what PCIe carries for this GPU right now, with nothing of the blend in it. Moves
 * `bytes` per iteration between pinned host memory and the device for about `seconds`:
 *   mode 0  copy engine, both directions at once (the best a staged path could do)
 *   mode 1  a kernel that reads and rewrites host memory in place (the zero-copy path's shape)
 * and returns GB/s per direction. Call it on every GPU at the same time to measure a box
 * (tools/pcie_ceiling.cu is the stand-alone version). */
FLUC_EXPORT int fluc_ttmlblend_pcie_probe (FlucTtmlBlend *thiz, int mode, size_t bytes, double seconds,
    double *gbs_per_direction);
/* The cudaStream_t the batched blend launches on, as an opaque pointer. */
FLUC_EXPORT void *fluc_ttmlblend_stream_handle (FlucTtmlBlend *thiz);

#ifdef __cplusplus
}
#endif
#endif /* _FLUC_TTMLBLEND_H_ */
