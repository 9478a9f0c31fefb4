/*
 * gstflucallocator.c -- GstAllocator handing out the context's pinned staging
 * frames (fluc_ttmlblend_frame_pool_acquire (..., on_host = 1, ...)).
 *
 * Part of the `-Dttml_cuda=enabled` build next to gstttmlblend.c (INTEGRATION.md). The graft
 * image has no GLib / GStreamer: there it is compiled and RUN against the functional fake in
 * tests/gst_stub/ (tests/test_gpu_gstglue.py).
 *
 * Why: fluc_ttmlblend_blend_host () blends device-accessible host memory
 * zero-copy -- the kernel reads the rows under the cue over PCIe and writes
 * them back, batched across streams -- while pageable memory has to be staged
 * by worker threads. ttmlblend proposes this allocator upstream in its
 * propose_allocation so that decoders / videotestsrc write their frames
 * straight into pinned pool frames. This is SURVEY.md section 8f rank 2, the
 * "device frame-buffer pool bridged to GstBuffer (pinned staging)" of
 * BASELINE.json's north_star. The memory is ordinary system memory to every
 * other element (GST_ALLOCATOR_SYSMEM-compatible map), so nothing else in a
 * pipeline has to know.
 */
#ifdef HAVE_CONFIG_H
#include "config.h"
#endif

#include "gstflucallocator.h"

#define GST_TYPE_FLUC_ALLOCATOR (gst_fluc_allocator_get_type ())
G_DECLARE_FINAL_TYPE (GstFlucAllocator, gst_fluc_allocator, GST, FLUC_ALLOCATOR, GstAllocator)

struct _GstFlucAllocator
{
  GstAllocator parent;
  FlucTtmlBlend *ctx;           /* not owned: lives as long as the element */
  GstVideoInfo info;
  FlucTtmlBlendFormat format;
};

typedef struct
{
  GstMemory mem;
  FlucTtmlBlendFrame frame;     /* pool frame: planes contiguous from plane[0] */
} GstFlucMemory;

G_DEFINE_TYPE (GstFlucAllocator, gst_fluc_allocator, GST_TYPE_ALLOCATOR);

static gsize
frame_size (GstFlucAllocator * self, const FlucTtmlBlendFrame * f)
{
  gsize size = 0;
  gint p;
  for (p = 0; p < fluc_ttmlblend_format_planes (self->format); p++)
    size += (gsize) f->stride[p] * fluc_ttmlblend_plane_rows (self->format, p,
        GST_VIDEO_INFO_HEIGHT (&self->info));
  return size;
}

static GstMemory *
gst_fluc_allocator_alloc (GstAllocator * allocator, gsize size, GstAllocationParams * params)
{
  GstFlucAllocator *self = GST_FLUC_ALLOCATOR (allocator);
  GstFlucMemory *mem = g_new0 (GstFlucMemory, 1);
  gsize real;

  if (fluc_ttmlblend_frame_pool_acquire (self->ctx, self->format,
          GST_VIDEO_INFO_WIDTH (&self->info), GST_VIDEO_INFO_HEIGHT (&self->info), 1,
          &mem->frame) != FLUC_TTMLBLEND_OK) {
    g_free (mem);
    return NULL;
  }
  real = frame_size (self, &mem->frame);
  if (real < size) {            /* caller wants more than one frame of this geometry */
    fluc_ttmlblend_frame_pool_release (self->ctx, &mem->frame);
    g_free (mem);
    return NULL;
  }
  gst_memory_init (GST_MEMORY_CAST (mem), 0, allocator, NULL, real, 255, 0, real);
  return GST_MEMORY_CAST (mem);
}

static void
gst_fluc_allocator_free (GstAllocator * allocator, GstMemory * memory)
{
  GstFlucAllocator *self = GST_FLUC_ALLOCATOR (allocator);
  GstFlucMemory *mem = (GstFlucMemory *) memory;
  fluc_ttmlblend_frame_pool_release (self->ctx, &mem->frame);   /* back to the pool, stays pinned */
  g_free (mem);
}

static gpointer
gst_fluc_memory_map (GstMemory * memory, gsize maxsize, GstMapFlags flags)
{
  return ((GstFlucMemory *) memory)->frame.plane[0];
}

static void
gst_fluc_memory_unmap (GstMemory * memory)
{
}

static void
gst_fluc_allocator_class_init (GstFlucAllocatorClass * klass)
{
  GstAllocatorClass *allocator_class = GST_ALLOCATOR_CLASS (klass);
  allocator_class->alloc = gst_fluc_allocator_alloc;
  allocator_class->free = gst_fluc_allocator_free;
}

static void
gst_fluc_allocator_init (GstFlucAllocator * self)
{
  GstAllocator *alloc = GST_ALLOCATOR_CAST (self);
  alloc->mem_type = "FlucPinnedFrame";
  alloc->mem_map = gst_fluc_memory_map;
  alloc->mem_unmap = gst_fluc_memory_unmap;
  GST_OBJECT_FLAG_SET (self, GST_ALLOCATOR_FLAG_CUSTOM_ALLOC);
}

/* The strides / offsets a buffer from this allocator must carry as GstVideoMeta
 * (pool frames use 256-byte multiple strides, not GStreamer's default 4). */
void
gst_fluc_allocator_fill_video_meta (GstAllocator * allocator, GstMemory * memory,
    gsize offset[GST_VIDEO_MAX_PLANES], gint stride[GST_VIDEO_MAX_PLANES])
{
  GstFlucAllocator *self = GST_FLUC_ALLOCATOR (allocator);
  GstFlucMemory *mem = (GstFlucMemory *) memory;
  gint p;
  for (p = 0; p < fluc_ttmlblend_format_planes (self->format); p++) {
    offset[p] = (guint8 *) mem->frame.plane[p] - (guint8 *) mem->frame.plane[0];
    stride[p] = mem->frame.stride[p];
  }
}

gboolean
gst_is_fluc_memory (GstMemory * memory)
{
  return memory->allocator != NULL && memory->allocator->mem_type != NULL &&
      strcmp (memory->allocator->mem_type, "FlucPinnedFrame") == 0;
}

GstBuffer *
gst_fluc_allocator_alloc_video_buffer (GstAllocator * allocator)
{
  GstFlucAllocator *self = GST_FLUC_ALLOCATOR (allocator);
  gsize offset[GST_VIDEO_MAX_PLANES] = { 0, };
  gint stride[GST_VIDEO_MAX_PLANES] = { 0, };
  GstMemory *mem = gst_allocator_alloc (allocator, 0, NULL);
  GstBuffer *buf;

  if (!mem)
    return NULL;
  buf = gst_buffer_new ();
  gst_buffer_append_memory (buf, mem);
  gst_fluc_allocator_fill_video_meta (allocator, mem, offset, stride);
  gst_buffer_add_video_meta_full (buf, GST_VIDEO_FRAME_FLAG_NONE, GST_VIDEO_INFO_FORMAT (&self->info),
      GST_VIDEO_INFO_WIDTH (&self->info), GST_VIDEO_INFO_HEIGHT (&self->info),
      fluc_ttmlblend_format_planes (self->format), offset, stride);
  return buf;
}

GstAllocator *
gst_fluc_allocator_new (FlucTtmlBlend * ctx, const GstVideoInfo * info, FlucTtmlBlendFormat format)
{
  GstFlucAllocator *self = g_object_new (GST_TYPE_FLUC_ALLOCATOR, NULL);
  self->ctx = ctx;
  self->info = *info;
  self->format = format;
  return GST_ALLOCATOR_CAST (gst_object_ref_sink (self));
}
