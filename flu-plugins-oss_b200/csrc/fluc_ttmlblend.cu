/*
 * fluc_ttmlblend.cu -- host side of libfluc_ttmlblend.so: the C ABI declared in
 * include/fluc_ttmlblend.h. Context (one per GPU), overlay cache, frame pool,
 * multi-stream batch scheduler and the host-frame (PCIe) path.
 *
 * This is the native runtime around the kernels in ttmlblend_kernels.cu. It
 * stands where the reference leaves compositing to GStreamer
 * (/root/reference/plugins/ttml/README.md:45-48) and is shaped after the
 * reference's own helper libraries: opaque object + monitor
 * (/root/reference/libs/fluc/flu-codec-sdk/fluc/threads/fluc_monitor.c:15-70),
 * worker thread draining a queue under that monitor
 * (/root/reference/libs/flu/downloader/lib/fludownloader.c:490-532), stats
 * copied out under the lock (.../bwmeter/fluc_bwmeter.c:71-76).
 *
 * No CPU fallback exists anywhere in this file: without a usable CUDA device
 * every entry point fails with FLUC_TTMLBLEND_ERROR_NO_DEVICE / _CUDA.
 */
#include "ttmlblend_internal.h"

#include <ctype.h>
#include <sched.h>

using namespace tbh;

struct _FlucTtmlBlend {
  Ctx c;
  uint32_t repeat_set = 0;      /* submit_many_repeat: next destination set */
};

#define ENTER(thiz)                                                          \
  if (!(thiz)) return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;                 \
  Ctx *c = &(thiz)->c;                                                       \
  std::unique_lock<std::mutex> lk (c->mu);                                   \
  if (c->sticky) return c->sticky;                                           \
  cudaSetDevice (c->device)

extern "C" {

const char *
fluc_ttmlblend_version (void)
{
  return "fluc_ttmlblend 0.1 (sm_100a)";
}

const char *
fluc_ttmlblend_strerror (int err)
{
  switch (err) {
    case FLUC_TTMLBLEND_OK: return "ok";
    case FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT: return "invalid argument";
    case FLUC_TTMLBLEND_ERROR_NO_DEVICE: return "no usable CUDA device (there is no CPU fallback)";
    case FLUC_TTMLBLEND_ERROR_CUDA: return "CUDA error (context unusable)";
    case FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY: return "out of memory";
    case FLUC_TTMLBLEND_ERROR_UNSUPPORTED_FORMAT: return "unsupported video format";
    case FLUC_TTMLBLEND_ERROR_NOT_FOUND: return "not found";
    case FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES: return "too many rectangles";
    default: return "unknown error";
  }
}

int
fluc_ttmlblend_device_count (void)
{
  int n = 0;
  if (cudaGetDeviceCount (&n) != cudaSuccess) {
    cudaGetLastError ();
    return 0;
  }
  return n;
}

/* The NUMA node of the GPU and its CPUs, from sysfs (Linux; silently nothing elsewhere). */
static void
find_numa_cpus (Ctx *c)
{
  const char *e = getenv ("FLUC_TTMLBLEND_NUMA");
  if (e && atoi (e) == 0)
    return;
  char bus[32] = "";
  if (cudaDeviceGetPCIBusId (bus, sizeof bus, c->device) != cudaSuccess) {
    cudaGetLastError ();
    return;
  }
  for (char *p = bus; *p; p++)
    *p = (char) tolower ((unsigned char) *p);
  char path[128];
  snprintf (path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE *f = fopen (path, "r");
  int node = -1;
  if (f) {
    if (fscanf (f, "%d", &node) != 1)
      node = -1;
    fclose (f);
  }
  if (node < 0)
    return;
  snprintf (path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
  f = fopen (path, "r");
  if (!f)
    return;
  char list[4096] = "";
  if (!fgets (list, sizeof list, f))
    list[0] = 0;
  fclose (f);
  for (char *tok = strtok (list, ",\n"); tok; tok = strtok (nullptr, ",\n")) {
    int a = -1, b = -1;
    if (sscanf (tok, "%d-%d", &a, &b) == 2) {
      for (int i = a; i <= b && i < CPU_SETSIZE; i++)
        c->numa_cpus.push_back (i);
    } else if (sscanf (tok, "%d", &a) == 1 && a < CPU_SETSIZE) {
      c->numa_cpus.push_back (a);
    }
  }
  if (!c->numa_cpus.empty ())
    c->numa_node = node;
  TBLOG (1, "device %d (%s) is on NUMA node %d, %zu CPUs", c->device, bus, node, c->numa_cpus.size ());
}

/* Runs the calling thread on the GPU's NUMA node for the lifetime of the object (first-touch /
 * local allocation policy then places pinned pages there); the previous affinity comes back. */
struct NumaScope {
  cpu_set_t old_set;
  bool moved = false;
  explicit NumaScope (const Ctx *c)
  {
    if (c->numa_cpus.empty () || sched_getaffinity (0, sizeof old_set, &old_set) != 0)
      return;
    cpu_set_t want;
    CPU_ZERO (&want);
    int n = 0;
    for (int cpu : c->numa_cpus)
      if (CPU_ISSET (cpu, &old_set)) {    /* stay inside what the process is allowed (cgroups, taskset) */
        CPU_SET (cpu, &want);
        n++;
      }
    if (n && sched_setaffinity (0, sizeof want, &want) == 0)
      moved = true;
  }
  ~NumaScope ()
  {
    if (moved)
      sched_setaffinity (0, sizeof old_set, &old_set);
  }
};

/* Streams, events and the memory pool fluc_ttmlblend_new creates (also its failure path). */
static void
destroy_cuda_objects (Ctx *c)
{
  for (cudaEvent_t &e : c->ev_fence)
    if (e) { cudaEventDestroy (e); e = nullptr; }
  for (cudaEvent_t *e : { &c->timer0, &c->timer1 })
    if (*e) { cudaEventDestroy (*e); *e = nullptr; }
  for (cudaStream_t *st : { &c->blend_stream, &c->up_stream, &c->reaper, &c->table_stream, &c->dma_in, &c->dma_out })
    if (*st) { cudaStreamDestroy (*st); *st = nullptr; }
  if (c->mem_pool) { cudaMemPoolDestroy (c->mem_pool); c->mem_pool = nullptr; }
}

int
fluc_ttmlblend_new (int device, FlucTtmlBlend **out)
{
  if (!out)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount (&n) != cudaSuccess || n <= 0) {
    cudaGetLastError ();
    return FLUC_TTMLBLEND_ERROR_NO_DEVICE;
  }
  if (device < 0) {
    const char *e = getenv ("FLUC_TTMLBLEND_DEVICE");
    device = e ? atoi (e) : 0;
  }
  if (device >= n)
    return FLUC_TTMLBLEND_ERROR_NO_DEVICE;
  if (cudaSetDevice (device) != cudaSuccess) {
    cudaGetLastError ();
    return FLUC_TTMLBLEND_ERROR_NO_DEVICE;
  }
  FlucTtmlBlend *t = new (std::nothrow) FlucTtmlBlend ();
  if (!t)
    return FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY;
  Ctx *c = &t->c;
  c->device = device;
  if (const char *sy = getenv ("FLUC_TTMLBLEND_SYNC"))
    c->blocking_sync = strcmp (sy, "block") == 0;
  bool ok = true;
  /* the copy streams of host DMA batches first */
  ok &= cudaStreamCreateWithFlags (&c->dma_in, cudaStreamNonBlocking) == cudaSuccess;
  ok &= cudaStreamCreateWithFlags (&c->dma_out, cudaStreamNonBlocking) == cudaSuccess;
  ok &= cudaStreamCreateWithFlags (&c->blend_stream, cudaStreamNonBlocking) == cudaSuccess;
  ok &= cudaStreamCreateWithFlags (&c->up_stream, cudaStreamNonBlocking) == cudaSuccess;
  ok &= cudaStreamCreateWithFlags (&c->reaper, cudaStreamNonBlocking) == cudaSuccess;
  ok &= cudaStreamCreateWithFlags (&c->table_stream, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < kDmaSets && ok; i++)
    ok &= cudaEventCreateWithFlags (&c->dma_sets[i].done, cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; i < 2 && ok; i++)
    ok &= cudaEventCreateWithFlags (&c->ev_fence[i], cudaEventDisableTiming) == cudaSuccess;
  ok &= cudaEventCreate (&c->timer0) == cudaSuccess;
  ok &= cudaEventCreate (&c->timer1) == cudaSuccess;
  if (ok) {
    /* a memory pool of our own for the stream-ordered overlay allocations: freed overlay
     * memory stays in it instead of going back to the OS, and nothing process-wide (the
     * device's default pool, which other libraries may use) is reconfigured */
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    ok &= cudaMemPoolCreate (&c->mem_pool, &props) == cudaSuccess;
    if (ok) {
      uint64_t thr = ~0ull;
      cudaMemPoolSetAttribute (c->mem_pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
  }
  if (!ok) {
    cudaGetLastError ();
    destroy_cuda_objects (c);
    delete t;
    return FLUC_TTMLBLEND_ERROR_NO_DEVICE;
  }
  const char *e;
  if ((e = getenv ("FLUC_TTMLBLEND_BATCH")))
    c->max_batch = (uint32_t) std::max (1, std::min (1024, atoi (e)));
  if ((e = getenv ("FLUC_TTMLBLEND_PROFILE_EVERY")))
    c->profile_every = (uint32_t) std::max (1, atoi (e));
  if ((e = getenv ("FLUC_TTMLBLEND_AUTOCROP")))
    c->autocrop = atoi (e) != 0;
  if ((e = getenv ("FLUC_TTMLBLEND_GROUPS")))
    c->use_groups = atoi (e) != 0;
  if ((e = getenv ("FLUC_TTMLBLEND_EAGER_PREPARE")))
    c->eager_prepare = atoi (e) != 0;
  if ((e = getenv ("FLUC_TTMLBLEND_MULTI")))
    c->use_multi = atoi (e) != 0;
  if ((e = getenv ("FLUC_TTMLBLEND_PDL")))
    c->use_pdl = atoi (e) != 0;
  if ((e = getenv ("FLUC_TTMLBLEND_HOST_DMA")))
    c->host_dma_policy = std::max (0, std::min (2, atoi (e)));
  if ((e = getenv ("FLUC_TTMLBLEND_DMA_PIECE")))
    c->dma_piece = (uint32_t) std::max (0, std::min (1024, atoi (e)));
  c->stage_threads = (int) std::max (2u, std::min (12u, std::thread::hardware_concurrency () * 3 / 4));
  if ((e = getenv ("FLUC_TTMLBLEND_STAGE_THREADS")))
    c->stage_threads = std::max (1, std::min (64, atoi (e)));
  if ((e = getenv ("FLUC_TTMLBLEND_STAGE_SLOTS")))
    c->stage_slots_max = std::max (1, std::min (4096, atoi (e)));
  if ((e = getenv ("FLUC_TTMLBLEND_AUTO_REGISTER")))
    c->auto_register = atoi (e) != 0;
  if ((e = getenv ("FLUC_TTMLBLEND_LINGER_US")))
    c->linger_us = (uint32_t) std::max (0, atoi (e));
  find_numa_cpus (c);
  c->sched = std::thread (scheduler_main, c);
  *out = t;
  TBLOG (1, "context on device %d", device);
  return 0;
}

void
fluc_ttmlblend_free (FlucTtmlBlend *thiz)
{
  if (!thiz)
    return;
  Ctx *c = &thiz->c;
  {
    std::unique_lock<std::mutex> lk (c->mu);
    c->quit = true;
    c->cv.notify_all ();
    c->launched_cv.notify_all ();
  }
  if (c->sched.joinable ())
    c->sched.join ();
  stage_shutdown (c);
  cudaSetDevice (c->device);
  if (!c->dma_trace.empty ()) {
    cudaDeviceSynchronize ();
    const size_t n = c->dma_trace.size (), a = n > 12 ? n - 12 : 0;
    for (size_t i = a; i < n; i++) {
      float t[4] = { 0, 0, 0, 0 };
      for (int k = 0; k < 4; k++)
        cudaEventElapsedTime (&t[k], c->dma_trace[a][0], c->dma_trace[i][k]);
      fprintf (stderr, "dma batch %zu: copy-in %.3f .. %.3f ms, copy-out %.3f .. %.3f ms\n", i, t[0], t[1], t[2], t[3]);
    }
  }
  /* our own streams only: other users of the device are none of our business */
  for (cudaStream_t st : { c->blend_stream, c->up_stream, c->table_stream, c->dma_in, c->dma_out })
    cudaStreamSynchronize (st);
  {
    std::unique_lock<std::mutex> lk (c->mu);
    c->pending.clear ();
    for (auto &b : c->batches) {
      if (b.t0) cudaEventDestroy (b.t0);
      if (b.t1) cudaEventDestroy (b.t1);
      cudaEventDestroy (b.done);
    }
    c->batches.clear ();
    c->overlays.clear ();       /* frees through the reaper stream */
    cudaStreamSynchronize (c->reaper);
    for (auto e : c->event_pool)
      cudaEventDestroy (e);
    for (auto e : c->timing_pool)
      cudaEventDestroy (e);
    auto free_slot = [](TableSlot &s) {
      if (s.h_jobs) cudaFreeHost (s.h_jobs);
      if (s.h_begin) cudaFreeHost (s.h_begin);
      if (s.d_jobs) cudaFree (s.d_jobs);
      if (s.d_begin) cudaFree (s.d_begin);
      if (s.copied) cudaEventDestroy (s.copied);
      if (s.uploaded) cudaEventDestroy (s.uploaded);
    };
    for (auto &s : c->slots)
      free_slot (s);
    stage_free_slots (c);
    for (auto &p : c->pool_free)
      if (!p.in_slab) {
        if (p.on_host) cudaFreeHost (p.base); else cudaFree (p.base);
      }
    for (auto &p : c->pool_used)
      if (!p.in_slab) {
        if (p.on_host) cudaFreeHost (p.base); else cudaFree (p.base);
      }
    for (void *slab : c->host_slabs)
      cudaFreeHost (slab);
    for (DmaSet &ds : c->dma_sets) {
      if (ds.dev) cudaFree (ds.dev);
      if (ds.done) cudaEventDestroy (ds.done);
    }
    for (auto &pair : c->dma_choice.ev)
      for (cudaEvent_t e : pair)
        if (e) cudaEventDestroy (e);
    for (auto &r : c->auto_regs)
      cudaHostUnregister ((void *) r.first);
    c->auto_regs.clear ();
    if (c->scrub) cudaFree (c->scrub);
    destroy_cuda_objects (c);
  }
  delete thiz;
}

int
fluc_ttmlblend_numa_node (FlucTtmlBlend *thiz)
{
  return thiz ? thiz->c.numa_node : -1;
}

const char *
fluc_ttmlblend_last_cuda_error (FlucTtmlBlend *thiz)
{
  if (!thiz)
    return "";
  /* a copy per calling thread: the context's own string changes under other threads' errors
   * once the lock is dropped */
  static thread_local std::string copy;
  std::unique_lock<std::mutex> lk (thiz->c.mu);
  copy = thiz->c.cuda_error;
  return copy.c_str ();
}

/* ---- overlay --------------------------------------------------------- */

int
fluc_ttmlblend_overlay_set_rectangles (FlucTtmlBlend *thiz, uint32_t stream,
    const FlucTtmlBlendRectangle *rects, uint32_t n_rects)
{
  ENTER (thiz);
  if (n_rects && !rects)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  if (n_rects > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  return overlay_install (c, lk, stream, rects, n_rects);
}

int
fluc_ttmlblend_overlay_set (FlucTtmlBlend *thiz, uint32_t stream, const uint8_t *bgra,
    int32_t w, int32_t h, int32_t stride, const FlucTtmlBlendRect *rects, uint32_t n_rects)
{
  ENTER (thiz);
  if (!bgra || w <= 0 || h <= 0 || stride < 4 * w || (n_rects && !rects))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  std::vector<FlucTtmlBlendRect> in;
  if (n_rects == 0) {
    in.push_back ({ 0, 0, w, h });
  } else {
    for (uint32_t i = 0; i < n_rects; i++) {
      /* region boxes clipped to the image ttmlrender drew them into */
      const int x0 = std::max (rects[i].x, 0), y0 = std::max (rects[i].y, 0);
      const int x1 = std::min (rects[i].x + rects[i].w, w), y1 = std::min (rects[i].y + rects[i].h, h);
      if (x1 > x0 && y1 > y0)
        in.push_back ({ x0, y0, x1 - x0, y1 - y0 });
    }
    in = disjoint_cover (in);
  }
  if (in.size () > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  std::vector<FlucTtmlBlendRectangle> rr;
  for (auto &r : in) {
    FlucTtmlBlendRectangle q = {};
    q.pixels = bgra + (size_t) r.y * stride + (size_t) r.x * 4;
    q.width = r.w;
    q.height = r.h;
    q.stride = stride;
    q.x = r.x;
    q.y = r.y;
    q.global_alpha = 1.0f;
    q.flags = FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA;   /* Cairo ARGB32, gstttmlrender.c:1446 */
    rr.push_back (q);
  }
  return overlay_install (c, lk, stream, rr.data (), (uint32_t) rr.size (), w, h);
}

int
fluc_ttmlblend_overlay_update (FlucTtmlBlend *thiz, uint32_t stream, const uint8_t *bgra,
    int32_t w, int32_t h, int32_t stride, const FlucTtmlBlendRect *changed, uint32_t n_changed)
{
  {
    ENTER (thiz);
    if (!bgra || w <= 0 || h <= 0 || stride < 4 * w || (n_changed && !changed))
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
    const int rc = overlay_update_image (c, lk, stream, bgra, w, h, stride, changed, n_changed);
    if (rc != FLUC_TTMLBLEND_ERROR_NOT_FOUND)
      return rc;
  }
  /* nothing to patch: the image whole (auto-crop finds what is in it) */
  return fluc_ttmlblend_overlay_set (thiz, stream, bgra, w, h, stride, nullptr, 0);
}

int
fluc_ttmlblend_overlay_set_regions (FlucTtmlBlend *thiz, uint32_t stream, int32_t W, int32_t H,
    const FlucTtmlBlendRegion *regions, uint32_t n_regions)
{
  ENTER (thiz);
  if (W <= 0 || H <= 0 || W > 32768 || H > 32768 || (n_regions && !regions))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  if (n_regions > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  return overlay_install_regions (c, lk, stream, W, H, regions, n_regions);
}

int
fluc_ttmlblend_overlay_clear (FlucTtmlBlend *thiz, uint32_t stream)
{
  ENTER (thiz);
  c->overlays.erase (stream);
  return 0;
}

int
fluc_ttmlblend_overlay_set_global_alpha (FlucTtmlBlend *thiz, uint32_t stream, const float *global_alpha, uint32_t n)
{
  ENTER (thiz);
  if (!global_alpha || n == 0 || n > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  int ga[FLUC_TTMLBLEND_MAX_RECTANGLES];
  for (uint32_t i = 0; i < n; i++) {
    if (!(global_alpha[i] >= 0.0f && global_alpha[i] <= 1.0f))     /* NaN fails both */
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
    ga[i] = (int) (255.0 * global_alpha[i]);        /* gst_video_blend, as overlay_set_rectangles */
  }
  return overlay_set_alpha (c, stream, ga, n);
}

int
fluc_ttmlblend_overlay_set_positions (FlucTtmlBlend *thiz, uint32_t stream, const int32_t *x, const int32_t *y,
    uint32_t n)
{
  ENTER (thiz);
  if (!x || !y)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  return overlay_set_positions (c, stream, x, y, n);
}

int
fluc_ttmlblend_overlay_set_render_rectangles (FlucTtmlBlend *thiz, uint32_t stream, const FlucTtmlBlendRect *render,
    uint32_t n)
{
  ENTER (thiz);
  if (!render)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  return overlay_set_render (c, lk, stream, render, n);
}

int
fluc_ttmlblend_set_chroma_mode (FlucTtmlBlend *thiz, int mode)
{
  ENTER (thiz);
  if (mode != FLUC_TTMLBLEND_CHROMA_SITED && mode != FLUC_TTMLBLEND_CHROMA_AVERAGE)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  c->chroma_average = mode == FLUC_TTMLBLEND_CHROMA_AVERAGE;
  return 0;
}

/* ---- device-resident frames ------------------------------------------ */

/* A frame joins the pending batch only if no queued frame conflicts with it: the CTAs of one
 * launch run in no particular order, so a frame that writes what a queued frame writes (the
 * same buffer twice) or reads (ping-pong pools), or reads what a queued frame writes (chained
 * overlays: stream A's output is stream B's input) has the batch launched first; launches on
 * the blend stream then run in order. Frames that only share a source are fine. */
static int
order_against_pending (Ctx *c, const FrameExtent &src, const FrameExtent &dst, bool inplace)
{
  if (c->pending.empty ())
    return 0;
  if (dst.hits (c->pending_dst) || dst.hits (c->pending_src) || (!inplace && src.hits (c->pending_dst)))
    return launch_pending (c);
  return 0;
}

static int
submit_locked (Ctx *c, uint32_t stream, int fmt, int32_t W, int32_t H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *src, const FlucTtmlBlendFrame *dst, uint64_t *ticket,
    const std::shared_ptr<StreamAfter> &after)
{
  int rc;
  fmt = format_canon (fmt);
  if ((rc = check_frame (fmt, W, H, src)) || (rc = check_frame (fmt, W, H, dst)))
    return rc;
  PendingFrame f;
  f.prep = nullptr;
  f.after = after;
  auto it = c->overlays.find (stream);
  if (it != c->overlays.end ()) {
    f.overlay = it->second;
    if ((rc = prepare_overlay (c, f.overlay.get (), fmt, W, H, &f.prep)))
      return rc;
    f.prep->used = true;
  }
  const bool inplace = src->plane[0] == dst->plane[0];
  const FrameExtent xs (fmt, W, H, src), xd (fmt, W, H, dst);
  if ((rc = order_against_pending (c, xs, xd, inplace)))
    return rc;
  f.layout = find_layout (c, f.prep, f.overlay && (inplace ? f.overlay->lazy_inplace : f.overlay->opaque_skip),
      fmt, W, H, frame_flags, src, dst, inplace);
  for (int pl = 0; pl < 3; pl++) {
    f.src[pl] = static_cast<const uint8_t *> (src->plane[pl]);
    f.dst[pl] = static_cast<uint8_t *> (dst->plane[pl]);
  }
  f.ticket = ++c->next_ticket;
  f.stream = stream;
  note_stream (c, stream);
  if (ticket)
    *ticket = f.ticket;
  if (c->pending.empty ())
    c->oldest_pending = std::chrono::steady_clock::now ();
  xd.add_to (c->pending_dst);
  if (!inplace)
    xs.add_to (c->pending_src);
  c->pending.push_back (std::move (f));
  if (c->pending.size () >= c->max_batch)
    return launch_pending (c);
  return 0;
}

int
fluc_ttmlblend_submit (FlucTtmlBlend *thiz, uint32_t stream, FlucTtmlBlendFormat fmt,
    int32_t W, int32_t H, uint32_t frame_flags, const FlucTtmlBlendFrame *src,
    const FlucTtmlBlendFrame *dst, uint64_t *ticket)
{
  ENTER (thiz);
  int rc = submit_locked (c, stream, fmt, W, H, frame_flags, src, dst, ticket, nullptr);
  if (rc == 0 && c->linger_us && !c->pending.empty ())
    c->cv.notify_all ();
  return rc;
}

static int
submit_many_locked (Ctx *c, uint32_t n, const uint32_t *streams, FlucTtmlBlendFormat fmt, int32_t W, int32_t H,
    uint32_t frame_flags, const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts, uint64_t *tickets,
    const std::shared_ptr<StreamAfter> &after)
{
  for (uint32_t i = 0; i < n; i++) {
    int rc = submit_locked (c, streams[i], fmt, W, H, frame_flags, &srcs[i], &dsts[i],
        tickets ? &tickets[i] : nullptr, after);
    if (rc)
      return rc;
  }
  if (c->linger_us && !c->pending.empty ())
    c->cv.notify_all ();
  return 0;
}

int
fluc_ttmlblend_submit_many (FlucTtmlBlend *thiz, uint32_t n, const uint32_t *streams,
    FlucTtmlBlendFormat fmt, int32_t W, int32_t H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts, uint64_t *tickets)
{
  ENTER (thiz);
  if (n && (!streams || !srcs || !dsts))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  return submit_many_locked (c, n, streams, fmt, W, H, frame_flags, srcs, dsts, tickets, nullptr);
}

/* A caller's CUDA stream (NULL: the legacy default stream of the context's device), which must
 * belong to the context's device: an event of one device cannot be recorded on, or waited for by,
 * a stream of another. */
static int
caller_stream (Ctx *c, void *cuda_stream, cudaStream_t *out)
{
  *out = cuda_stream ? static_cast<cudaStream_t> (cuda_stream) : cudaStreamLegacy;
  int dev = -1;
  if (cudaStreamGetDevice (*out, &dev) != cudaSuccess) {
    cudaGetLastError ();
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  }
  return dev == c->device ? 0 : FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
}

int
fluc_ttmlblend_submit_many_after (FlucTtmlBlend *thiz, void *cuda_stream, uint32_t n,
    const uint32_t *streams, FlucTtmlBlendFormat fmt, int32_t W, int32_t H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts, uint64_t *tickets)
{
  ENTER (thiz);
  if (n && (!streams || !srcs || !dsts))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  cudaStream_t st;
  int rc = caller_stream (c, cuda_stream, &st);
  if (rc || n == 0)
    return rc;
  /* declared after lk: goes back to the pool (when no frame holds it any more) under the lock */
  std::shared_ptr<StreamAfter> after (new StreamAfter ());
  after->ctx = c;
  after->ev = event_get (c);
  CU (c, cudaEventRecord (after->ev, st));
  return submit_many_locked (c, n, streams, fmt, W, H, frame_flags, srcs, dsts, tickets, after);
}

int
fluc_ttmlblend_submit_many_repeat (FlucTtmlBlend *thiz, uint32_t n, const uint32_t *streams,
    FlucTtmlBlendFormat fmt, int32_t W, int32_t H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *srcs, const FlucTtmlBlendFrame *dsts, uint32_t dst_sets, uint32_t repeats)
{
  if (!thiz || dst_sets == 0)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  uint32_t &set = thiz->repeat_set;      /* carries on where the previous call stopped */
  for (uint32_t r = 0; r < repeats; r++, set++) {
    int rc = fluc_ttmlblend_submit_many (thiz, n, streams, fmt, W, H, frame_flags, srcs,
        dsts + (size_t) (set % dst_sets) * n, nullptr);
    if (rc == 0)
      rc = fluc_ttmlblend_flush (thiz);
    if (rc)
      return rc;
  }
  return 0;
}

int
fluc_ttmlblend_flush (FlucTtmlBlend *thiz)
{
  ENTER (thiz);
  return launch_pending (c);
}

/* wait () and wait_on_stream () of a ticket that is not a staged host frame's: launches it if it is
 * still queued, then finds the `done` event of its batch (*ev = nullptr: finished). *failed: the
 * error of a batch whose launch failed half way. */
static int
launch_and_find (Ctx *c, std::unique_lock<std::mutex> &lk, uint64_t ticket, cudaEvent_t *ev, int *failed)
{
  *ev = nullptr;
  *failed = 0;
  if (!c->pending.empty () && ticket >= c->pending.front ().ticket) {
    /* The frame has not been launched yet. A lone stream launches now (lowest latency). When
     * several streams are active -- many elements calling blend + wait from their own
     * streaming threads -- the batch is left to the scheduler thread for up to the linger
     * time (or until it is full), so that the other streams' frames share the launch. */
    if (c->linger_us && several_streams_active (c) && c->pending.size () < c->max_batch) {
      c->cv.notify_all ();
      c->launched_cv.wait (lk, [&] {
        return c->quit || c->sticky || c->linger_us == 0 || c->pending.empty () ||
            ticket < c->pending.front ().ticket;
      });
      if (c->sticky)
        return c->sticky;
    }
    if (!c->pending.empty () && ticket >= c->pending.front ().ticket) {
      int rc = launch_pending (c);
      if (rc)
        return rc;
    }
  }
  /* a batch whose launch failed half way: still synchronise with what went out, then say so */
  for (const Ctx::FailedRange &fr : c->failed_ranges)
    if (ticket >= fr.first && ticket <= fr.last)
      *failed = fr.rc;
  /* a ticket whose batch has been retired is finished; it must not fall through to the next batch
   * in flight (a caller that waits one batch behind would then wait for the newest one) */
  if (ticket > c->retired_through)
    for (auto &b : c->batches)
      if (b.last_ticket >= ticket) {
        *ev = b.done;
        break;
      }
  return 0;
}

int
fluc_ttmlblend_wait (FlucTtmlBlend *thiz, uint64_t ticket)
{
  ENTER (thiz);
  if (ticket == 0 || ticket > c->next_ticket)
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  int staged_rc = 0;
  if (stage_wait (c, lk, ticket, &staged_rc))
    return staged_rc;
  cudaEvent_t ev;
  int failed;
  int rc = launch_and_find (c, lk, ticket, &ev, &failed);
  if (rc)
    return rc;
  if (!ev) {
    return failed;              /* already reaped: finished */
  }
  /* the event stays valid while we wait: batches are only reaped under mu,
   * and a reaped event goes back to the pool, not destroyed */
  lk.unlock ();
  cudaError_t e = cudaEventSynchronize (ev);
  lk.lock ();
  if (e != cudaSuccess) {
    c->sticky = FLUC_TTMLBLEND_ERROR_CUDA;
    c->cuda_error = std::string ("wait: ") + cudaGetErrorString (e);
    return c->sticky;
  }
  reap_batches (c);
  return failed;
}

int
fluc_ttmlblend_wait_on_stream (FlucTtmlBlend *thiz, uint64_t ticket, void *cuda_stream)
{
  ENTER (thiz);
  if (ticket == 0 || ticket > c->next_ticket)
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  cudaStream_t st;
  int rc = caller_stream (c, cuda_stream, &st);
  if (rc)
    return rc;
  /* a staged host frame is finished by a CPU copy, which no stream can wait for */
  if (c->stage_jobs.count (ticket))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  cudaEvent_t ev;
  int failed;
  if ((rc = launch_and_find (c, lk, ticket, &ev, &failed)))
    return rc;
  if (ev)
    CU (c, cudaStreamWaitEvent (st, ev, 0));
  return failed;
}

int
fluc_ttmlblend_sync (FlucTtmlBlend *thiz)
{
  ENTER (thiz);
  stage_drain (c, lk, 0);       /* staged host frames: every copy-in has reached the batch */
  int rc = launch_pending (c);
  if (rc)
    return rc;
  /* what is in flight now, then wait for it with the context unlocked: other threads keep
   * submitting frames and changing cues meanwhile (their work is not waited for) */
  const cudaStream_t streams[3] = { c->blend_stream, c->up_stream, c->dma_out };
  cudaEvent_t ev[3];
  int n_ev = 0;
  for (cudaStream_t st : streams) {
    cudaEvent_t e = event_get (c);
    CU (c, cudaEventRecord (e, st));
    ev[n_ev++] = e;
  }
  lk.unlock ();
  cudaError_t err = cudaSuccess;
  for (int i = 0; i < n_ev; i++) {
    const cudaError_t e = cudaEventSynchronize (ev[i]);
    err = err == cudaSuccess ? e : err;
  }
  lk.lock ();
  for (int i = 0; i < n_ev; i++)
    c->event_pool.push_back (ev[i]);
  if (err != cudaSuccess) {
    c->sticky = FLUC_TTMLBLEND_ERROR_CUDA;
    c->cuda_error = std::string ("sync: ") + cudaGetErrorString (err);
    return c->sticky;
  }
  reap_batches (c);
  stage_drain (c, lk, 1);       /* ... and has been copied back into the caller's frame */
  return c->sticky;
}

int
fluc_ttmlblend_set_batch (FlucTtmlBlend *thiz, uint32_t max_frames, uint32_t linger_us)
{
  ENTER (thiz);
  if (max_frames < 1 || max_frames > 1024)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  c->max_batch = max_frames;
  c->linger_us = linger_us;
  c->cv.notify_all ();
  c->launched_cv.notify_all ();
  return 0;
}

/* ---- host-resident frames -------------------------------------------- */

/* Everything of ours that may still touch host memory has finished: queued frames launched,
 * blend stream and host DMA copy streams drained. Needed before a registration goes away. */
static void
drain_host_users (Ctx *c)
{
  launch_pending (c);
  cudaStreamSynchronize (c->blend_stream);
  cudaStreamSynchronize (c->dma_in);
  cudaStreamSynchronize (c->dma_out);
}

/* How many automatic plane registrations are kept: a pool's worth of buffers (16) times three
 * planes for every stream that uses them, at least 192. */
static size_t
auto_reg_limit (const Ctx *c)
{
  return std::max<size_t> (192, std::min<size_t> (8192, 48 * c->auto_streams.size ()));
}

/* Opt-in (fluc_ttmlblend_set_auto_register): pin the memory of pageable host frames the
 * first time they are seen, so that later frames from the same buffers -- GStreamer buffer
 * pools recycle them -- take the zero-copy path (10.7 k instead of 1.7 k 4K frames/s,
 * tools/pageable_probe.py). Least recently used plane registrations are dropped beyond the limit.
 * The owner of the memory must call host_forget / host_unregister before it frees it: a
 * registration pins the physical pages, and a later allocation at the same address would be
 * taken for the registered one while the GPU still reaches the old pages. */
static void
auto_register_frame (Ctx *c, uint32_t stream, int fmt, int W, int H, const FlucTtmlBlendFrame *hf)
{
  /* range by range: planes that are neighbours in memory (GStreamer's default layout: one
   * memory per frame) are pinned as one range -- two registrations may not share a page --
   * while planes in allocations of their own get one each */
  const FrameExtent x (fmt, W, H, hf);
  for (int r = 0; r < x.n; r++) {
    const uintptr_t lo = x.lo[r], hi = x.hi[r];
    auto it = c->auto_regs.upper_bound (lo);
    if (it != c->auto_regs.begin ()) {
      --it;
      if (it->first <= lo && hi <= it->second.hi) {
        it->second.tick = ++c->auto_tick;      /* known: now most recently used */
        continue;
      }
    }
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes (&attr, (void *) lo) == cudaSuccess && attr.type == cudaMemoryTypeHost)
      continue;                 /* already pinned by someone else */
    cudaGetLastError ();
    c->auto_streams.insert (stream);
    if (c->auto_regs.size () >= auto_reg_limit (c)) {
      /* nothing queued or in flight may still use the oldest one */
      drain_host_users (c);
      auto oldest = c->auto_regs.begin ();
      for (auto k = c->auto_regs.begin (); k != c->auto_regs.end (); ++k)
        if (k->second.tick < oldest->second.tick)
          oldest = k;
      cudaHostUnregister ((void *) oldest->first);
      c->auto_regs.erase (oldest);
    }
    void *dev = nullptr;
    if (cudaHostRegister ((void *) lo, hi - lo, cudaHostRegisterDefault) == cudaSuccess) {
      if (cudaHostGetDevicePointer (&dev, (void *) lo, 0) == cudaSuccess)
        c->auto_regs[lo] = { hi, ++c->auto_tick, (uintptr_t) dev };
      else {
        cudaGetLastError ();
        cudaHostUnregister ((void *) lo);
      }
    } else
      cudaGetLastError ();      /* cannot pin (memlock limit, odd mapping): staged copies it is */
  }
}

int
fluc_ttmlblend_set_auto_register (FlucTtmlBlend *thiz, int enabled)
{
  ENTER (thiz);
  c->auto_register = enabled != 0;
  return 0;
}

int
fluc_ttmlblend_set_host_dma (FlucTtmlBlend *thiz, int mode)
{
  ENTER (thiz);
  if (mode < 0 || mode > 2)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  /* what is queued goes out the way it was queued for */
  if (!c->pending.empty ()) {
    int rc = launch_pending (c);
    if (rc)
      return rc;
  }
  c->host_dma_policy = mode;
  if (mode == 2) {
    /* measure afresh (the events are kept) */
    Ctx::DmaChoice &d = c->dma_choice;
    d.phase = 0;
    d.dma = false;
    d.judged = true;
    d.begun[0] = d.begun[1] = d.ended[0] = d.ended[1] = false;
  }
  return 0;
}


}  /* extern "C" */

/* A device-accessible host frame (zf: its device addresses, hf: its host addresses) joins the
 * pending batch: the blend kernel reads the rows under the cue from host memory and writes them
 * back, all over PCIe, one launch for every queued frame. Context locked. */
int
tbh::queue_mapped_frame (Ctx *c, uint64_t tk, uint32_t stream, const std::shared_ptr<Overlay> &ov, Prepared *prep,
    int fmt, int W, int H, uint32_t frame_flags, const FlucTtmlBlendFrame *zfp, const FlucTtmlBlendFrame *hf)
{
  int rc;
  const FlucTtmlBlendFrame &zf = *zfp;
  PendingFrame f;
  f.overlay = ov;
  f.prep = prep;
  f.ticket = tk;
  f.stream = stream;
  note_stream (c, stream);
  const FrameExtent xz (fmt, W, H, &zf), xh (fmt, W, H, hf);
  f.host = true;
  f.host_lo = xz.hull_lo ();
  f.host_hi = xz.hull_hi ();
  if ((rc = order_against_pending (c, xz, xz, true)))
    return rc;
  f.layout = find_layout (c, prep, ov->lazy_inplace, fmt, W, H, frame_flags, &zf, &zf, true);
  for (int pl = 0; pl < 3; pl++) {
    f.src[pl] = static_cast<const uint8_t *> (zf.plane[pl]);
    f.dst[pl] = static_cast<uint8_t *> (zf.plane[pl]);
  }
  xz.add_to (c->pending_dst);
  if (zf.plane[0] != hf->plane[0])
    xh.add_to (c->pending_dst);         /* no unified addressing: known under both addresses */
  xh.add_to (c->inflight_host);
  c->stats.h2d_bytes += f.layout->window_bytes;
  c->stats.d2h_bytes += f.layout->window_bytes;
  if (c->pending.empty ())
    c->oldest_pending = std::chrono::steady_clock::now ();
  c->pending.push_back (std::move (f));
  /* frames for the copy engines go out in pieces: the copy-out of one piece overlaps the copy-in of
   * the next inside one call as well, whatever the caller's own look-behind is */
  const bool pieces = c->dma_piece >= 4 && c->host_dma_policy != 0 && c->dma_now () &&
      c->pending.front ().host && layout_takes_dma (c->pending.front ().layout);
  const size_t full = pieces ? std::min<size_t> (c->max_batch, c->dma_piece) : c->max_batch;
  if (c->pending.size () >= full)
    return launch_pending (c);
  if (c->linger_us)
    c->cv.notify_all ();
  return 0;
}

extern "C" {

static int
blend_host_locked (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, int fmt, int32_t W, int32_t H,
    uint32_t frame_flags, const FlucTtmlBlendFrame *hf, uint64_t *ticket)
{
  int rc;
  fmt = format_canon (fmt);
  if ((rc = check_frame (fmt, W, H, hf)))
    return rc;
  const uint64_t tk = ++c->next_ticket;
  if (ticket)
    *ticket = tk;
  auto it = c->overlays.find (stream);
  if (it == c->overlays.end ())
    return 0;                   /* no overlay: the frame passes through untouched */
  std::shared_ptr<Overlay> ov = it->second;
  Prepared *prep = nullptr;
  if ((rc = prepare_overlay (c, ov.get (), fmt, W, H, &prep)))
    return rc;
  prep->used = true;

  /* Is the host frame device-accessible (pool frame / host_register)? Then the
   * kernel can reach it over PCIe itself. */
  const int n_planes = format_planes (fmt);
  if (c->auto_register)
    auto_register_frame (c, stream, fmt, W, H, hf);
  FlucTtmlBlendFrame zf = {};
  bool mapped = true;
  for (int pl = 0; pl < n_planes && mapped; pl++) {
    /* pinned pool frames are known (cudaHostAlloc under UVA: device pointer == host pointer):
     * no driver call per plane per frame for them */
    if (c->pinned_planes.count (hf->plane[pl])) {
      zf.plane[pl] = hf->plane[pl];
      zf.stride[pl] = hf->stride[pl];
      if ((zf.stride[pl] & 15) != 0)
        mapped = false;
      continue;
    }
    const uintptr_t lo = (uintptr_t) hf->plane[pl];
    const uintptr_t hi = lo + (uintptr_t) hf->stride[pl] * (uintptr_t) (plane_rows (fmt, pl, H) - 1) +
        (uintptr_t) plane_row_bytes (fmt, pl, W);
    /* planes this context registered itself are known too, with their whole range */
    auto ar = c->auto_regs.upper_bound (lo);
    if (ar != c->auto_regs.begin () && (--ar)->first <= lo && hi <= ar->second.hi) {
      zf.plane[pl] = (void *) (ar->second.dev + (lo - ar->first));
      zf.stride[pl] = hf->stride[pl];
      if ((((uintptr_t) zf.plane[pl] | (uintptr_t) zf.stride[pl]) & 15u) != 0)
        mapped = false;
      continue;
    }
    /* anything else: ask the driver, for the first and for the last byte of the plane (a
     * registration that ends inside the plane must not count) */
    cudaPointerAttributes attr, attr_end;
    if (cudaPointerGetAttributes (&attr, hf->plane[pl]) != cudaSuccess ||
        attr.type != cudaMemoryTypeHost || !attr.devicePointer ||
        cudaPointerGetAttributes (&attr_end, (const void *) (hi - 1)) != cudaSuccess ||
        attr_end.type != cudaMemoryTypeHost || !attr_end.devicePointer ||
        (uintptr_t) attr_end.devicePointer - (uintptr_t) attr.devicePointer != hi - 1 - lo) {
      cudaGetLastError ();
      mapped = false;
    } else {
      zf.plane[pl] = attr.devicePointer;
      zf.stride[pl] = hf->stride[pl];
      /* byte-granular accesses to host memory would each cross PCIe: frames that are not
       * 16-byte aligned go through the staging threads (copies into an aligned pinned frame) instead */
      if ((((uintptr_t) zf.plane[pl] | (uintptr_t) zf.stride[pl]) & 15u) != 0)
        mapped = false;
    }
  }

  if (mapped)
    return queue_mapped_frame (c, tk, stream, ov, prep, fmt, W, H, frame_flags, &zf, hf);

  /* Not device-accessible (ordinary pageable memory, or not 16-byte aligned): worker threads copy
   * the rows under the cue into a pinned staging frame, that frame is blended zero copy like
   * any other, and the rows are copied back (staging.cu). */
  return stage_frame (c, lk, tk, stream, ov, prep, fmt, W, H, frame_flags, hf);
}

int
fluc_ttmlblend_blend_host (FlucTtmlBlend *thiz, uint32_t stream, FlucTtmlBlendFormat fmt,
    int32_t W, int32_t H, uint32_t frame_flags, const FlucTtmlBlendFrame *hf, uint64_t *ticket)
{
  ENTER (thiz);
  return blend_host_locked (c, lk, stream, fmt, W, H, frame_flags, hf, ticket);
}

int
fluc_ttmlblend_blend_host_many (FlucTtmlBlend *thiz, uint32_t n, const uint32_t *streams,
    FlucTtmlBlendFormat fmt, int32_t W, int32_t H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *host_frames, uint64_t *tickets)
{
  ENTER (thiz);
  if (n && (!streams || !host_frames))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  for (uint32_t i = 0; i < n; i++) {
    int rc = blend_host_locked (c, lk, streams[i], fmt, W, H, frame_flags, &host_frames[i],
        tickets ? &tickets[i] : nullptr);
    if (rc)
      return rc;
  }
  return 0;
}

int
fluc_ttmlblend_host_register (FlucTtmlBlend *thiz, void *ptr, size_t bytes)
{
  ENTER (thiz);
  if (!ptr || !bytes)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  cudaError_t e = cudaHostRegister (ptr, bytes, cudaHostRegisterDefault);
  if (e != cudaSuccess) {
    cudaGetLastError ();
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  }
  return 0;
}

int
fluc_ttmlblend_host_unregister (FlucTtmlBlend *thiz, void *ptr)
{
  ENTER (thiz);
  /* frames of this memory may be queued or on the bus */
  drain_host_users (c);
  c->auto_regs.erase ((uintptr_t) ptr);
  cudaError_t e = cudaHostUnregister (ptr);
  if (e != cudaSuccess) {
    cudaGetLastError ();
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  }
  return 0;
}

int
fluc_ttmlblend_host_forget (FlucTtmlBlend *thiz, const void *ptr, size_t bytes)
{
  ENTER (thiz);
  if (!ptr || !bytes)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  const uintptr_t lo = (uintptr_t) ptr, hi = lo + bytes;
  bool drained = false;
  int n = 0;
  for (auto it = c->auto_regs.begin (); it != c->auto_regs.end ();) {
    if (it->first < hi && lo < it->second.hi) {
      if (!drained) {
        drain_host_users (c);
        drained = true;
      }
      if (cudaHostUnregister ((void *) it->first) != cudaSuccess)
        cudaGetLastError ();
      it = c->auto_regs.erase (it);
      n++;
    } else {
      ++it;
    }
  }
  return n;
}

/* ---- frame pool ------------------------------------------------------ */

int
fluc_ttmlblend_format_planes (FlucTtmlBlendFormat fmt)
{
  fmt = (FlucTtmlBlendFormat) format_canon (fmt);
  return format_valid (fmt) ? format_planes (fmt) : 0;
}

int
fluc_ttmlblend_plane_row_bytes (FlucTtmlBlendFormat fmt, int plane, int32_t width)
{
  fmt = (FlucTtmlBlendFormat) format_canon (fmt);
  if (!format_valid (fmt) || plane < 0 || plane >= format_planes (fmt))
    return 0;
  return plane_row_bytes (fmt, plane, width);
}

int
fluc_ttmlblend_plane_rows (FlucTtmlBlendFormat fmt, int plane, int32_t height)
{
  fmt = (FlucTtmlBlendFormat) format_canon (fmt);
  if (!format_valid (fmt) || plane < 0 || plane >= format_planes (fmt))
    return 0;
  return plane_rows (fmt, plane, height);
}

/* free frames are kept in address order, so that frames acquired one after the other are
 * neighbours in their slab */
static void
pool_free_insert (Ctx *c, const PoolEntry &e)
{
  auto pos = std::lower_bound (c->pool_free.begin (), c->pool_free.end (), e,
      [](const PoolEntry &a, const PoolEntry &b) { return (uintptr_t) a.base < (uintptr_t) b.base; });
  c->pool_free.insert (pos, e);
}

int
fluc_ttmlblend_frame_pool_acquire (FlucTtmlBlend *thiz, FlucTtmlBlendFormat fmt, int32_t W,
    int32_t H, int on_host, FlucTtmlBlendFrame *out)
{
  ENTER (thiz);
  fmt = (FlucTtmlBlendFormat) format_canon (fmt);
  if (!out || W <= 0 || H <= 0)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  if (!format_valid (fmt))
    return FLUC_TTMLBLEND_ERROR_UNSUPPORTED_FORMAT;
  on_host = on_host ? 1 : 0;
  for (size_t i = 0; i < c->pool_free.size (); i++) {
    PoolEntry &p = c->pool_free[i];
    if (p.fmt == fmt && p.W == W && p.H == H && p.on_host == on_host) {
      *out = p.frame;
      c->pool_used.push_back (p);
      c->pool_free.erase (c->pool_free.begin () + i);
      return 0;
    }
  }
  PoolEntry p = {};
  p.fmt = fmt; p.W = W; p.H = H; p.on_host = on_host;
  size_t off = 0, plane_off[3] = { 0, 0, 0 };
  const int n_planes = format_planes (fmt);
  for (int pl = 0; pl < n_planes; pl++) {
    p.frame.stride[pl] = (int32_t) align_up ((size_t) plane_row_bytes (fmt, pl, W), 256);
    plane_off[pl] = off;
    off += (size_t) p.frame.stride[pl] * plane_rows (fmt, pl, H);
  }
  p.bytes = off;
  if (on_host) {
    /* a slab of frames at a constant spacing: 4 the first time, then as many as the pool already
     * holds of this geometry (doubling), at most 32 frames or 512 MB */
    size_t have = 0;
    for (const PoolEntry &q : c->pool_used)
      have += (q.on_host && q.fmt == fmt && q.W == W && q.H == H) ? 1 : 0;
    size_t k = std::max<size_t> (4, std::min<size_t> (32, have));
    k = std::max<size_t> (1, std::min<size_t> (k, ((size_t) 512 << 20) / off));
    void *slab = nullptr;
    {
      NumaScope numa (c);       /* pages next to the GPU's PCIe root */
      CU (c, cudaHostAlloc (&slab, off * k, cudaHostAllocDefault));
    }
    c->host_slabs.push_back (slab);
    /* the first frame goes to the caller, the others wait in the pool in address order */
    for (size_t i = k; i-- > 0;) {
      PoolEntry q = p;
      q.in_slab = true;
      q.base = static_cast<uint8_t *> (slab) + i * off;
      for (int pl = 0; pl < n_planes; pl++) {
        q.frame.plane[pl] = static_cast<uint8_t *> (q.base) + plane_off[pl];
        c->pinned_planes.insert (q.frame.plane[pl]);
      }
      if (i == 0) {
        *out = q.frame;
        c->pool_used.push_back (q);
      } else {
        pool_free_insert (c, q);
      }
    }
    return 0;
  }
  CU (c, cudaMalloc (&p.base, off));
  for (int pl = 0; pl < n_planes; pl++)
    p.frame.plane[pl] = static_cast<uint8_t *> (p.base) + plane_off[pl];
  *out = p.frame;
  c->pool_used.push_back (p);
  return 0;
}

int
fluc_ttmlblend_frame_pool_release (FlucTtmlBlend *thiz, const FlucTtmlBlendFrame *frame)
{
  ENTER (thiz);
  if (!frame)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  for (size_t i = 0; i < c->pool_used.size (); i++)
    if (c->pool_used[i].frame.plane[0] == frame->plane[0]) {
      const PoolEntry e = c->pool_used[i];
      c->pool_used.erase (c->pool_used.begin () + i);
      pool_free_insert (c, e);
      return 0;
    }
  return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
}

static int
frame_copy (Ctx *c, int fmt, int W, int H, const FlucTtmlBlendFrame *s, const FlucTtmlBlendFrame *d,
    cudaMemcpyKind kind)
{
  int rc;
  fmt = format_canon (fmt);
  if ((rc = check_frame (fmt, W, H, s)) || (rc = check_frame (fmt, W, H, d)))
    return rc;
  for (int pl = 0; pl < format_planes (fmt); pl++) {
    const size_t rb = (size_t) plane_row_bytes (fmt, pl, W);
    CU (c, cudaMemcpy2DAsync (d->plane[pl], d->stride[pl], s->plane[pl], s->stride[pl], rb,
            plane_rows (fmt, pl, H), kind, c->blend_stream));
    if (kind == cudaMemcpyHostToDevice)
      c->stats.h2d_bytes += rb * plane_rows (fmt, pl, H);
    else
      c->stats.d2h_bytes += rb * plane_rows (fmt, pl, H);
  }
  CU (c, cudaStreamSynchronize (c->blend_stream));
  return 0;
}

int
fluc_ttmlblend_frame_upload (FlucTtmlBlend *thiz, FlucTtmlBlendFormat fmt, int32_t W, int32_t H,
    const FlucTtmlBlendFrame *host_src, const FlucTtmlBlendFrame *dev_dst)
{
  ENTER (thiz);
  return frame_copy (c, fmt, W, H, host_src, dev_dst, cudaMemcpyHostToDevice);
}

int
fluc_ttmlblend_frame_download (FlucTtmlBlend *thiz, FlucTtmlBlendFormat fmt, int32_t W, int32_t H,
    const FlucTtmlBlendFrame *dev_src, const FlucTtmlBlendFrame *host_dst)
{
  ENTER (thiz);
  int rc = launch_pending (c);
  if (rc)
    return rc;
  return frame_copy (c, fmt, W, H, dev_src, host_dst, cudaMemcpyDeviceToHost);
}

/* ---- outline blur (per cue, producer side) --------------------------- */

int
fluc_ttmlblend_blur_argb32 (FlucTtmlBlend *thiz, const uint8_t *src, int32_t w, int32_t h,
    int32_t stride, int32_t radius, double sigma, uint8_t *dst, int32_t dst_stride)
{
  ENTER (thiz);
  if (!src || !dst || w <= 0 || h <= 0 || stride < 4 * w || dst_stride < 4 * w || radius < 0 ||
      radius > 64 || !(sigma > 0.0))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  /* gst_ttml_blur_create_gaussian_kernel, /root/reference/plugins/ttml/gstttmlblur.c:28-67:
   * G(x,y) = exp (-(x^2 + y^2) / (2 sigma^2)) / (2 pi sigma^2), normalised, 16.16 fixed */
  const int size = 2 * radius + 1, n = size * size;
  std::vector<double> tmp (n);
  std::vector<int32_t> taps (n);
  const double scale2 = 2.0 * sigma * sigma;
  const double scale1 = 1.0 / (3.14159265358979323846 * scale2);
  double sum = 0;
  int i = 0;
  for (int x = -radius; x <= radius; ++x)
    for (int y = -radius; y <= radius; ++y, ++i) {
      const double u = x * x, v = y * y;
      tmp[i] = scale1 * exp (-(u + v) / scale2);
      sum += tmp[i];
    }
  for (i = 0; i < n; ++i)
    taps[i] = (int32_t) ((tmp[i] / sum) * 65536.0);       /* pixman_double_to_fixed */

  const size_t pitch = align_up ((size_t) w * 4, 256);
  void *d_src = nullptr, *d_dst = nullptr, *d_taps = nullptr;
  CU (c, cudaMallocFromPoolAsync (&d_src, pitch * h, c->mem_pool, c->up_stream));
  CU (c, cudaMallocFromPoolAsync (&d_dst, pitch * h, c->mem_pool, c->up_stream));
  CU (c, cudaMallocFromPoolAsync (&d_taps, (size_t) n * 4, c->mem_pool, c->up_stream));
  CU (c, cudaMemcpy2DAsync (d_src, pitch, src, stride, (size_t) w * 4, h, cudaMemcpyHostToDevice, c->up_stream));
  CU (c, cudaMemcpyAsync (d_taps, taps.data (), (size_t) n * 4, cudaMemcpyHostToDevice, c->up_stream));
  CU (c, launch_blur (static_cast<uint8_t *> (d_src), w, h, (int) pitch, static_cast<int32_t *> (d_taps),
          radius, static_cast<uint8_t *> (d_dst), (int) pitch, c->up_stream));
  CU (c, cudaMemcpy2DAsync (dst, dst_stride, d_dst, pitch, (size_t) w * 4, h, cudaMemcpyDeviceToHost, c->up_stream));
  CU (c, cudaFreeAsync (d_src, c->up_stream));
  CU (c, cudaFreeAsync (d_dst, c->up_stream));
  CU (c, cudaFreeAsync (d_taps, c->up_stream));
  CU (c, cudaStreamSynchronize (c->up_stream));
  c->stats.h2d_bytes += (uint64_t) w * 4 * h;
  c->stats.d2h_bytes += (uint64_t) w * 4 * h;
  return 0;
}

/* ---- several GPUs in one process -------------------------------------- */

struct _FlucTtmlBlendMulti {
  std::vector<FlucTtmlBlend *> ctx;
  std::vector<int> device;
};

int
fluc_ttmlblend_multi_new (const int *devices, uint32_t n_devices, FlucTtmlBlendMulti **out)
{
  if (!out)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  *out = nullptr;
  std::vector<int> devs;
  if (devices && n_devices) {
    devs.assign (devices, devices + n_devices);
  } else {
    const int n = fluc_ttmlblend_device_count ();
    for (int i = 0; i < n; i++)
      devs.push_back (i);
  }
  if (devs.empty ())
    return FLUC_TTMLBLEND_ERROR_NO_DEVICE;
  FlucTtmlBlendMulti *m = new (std::nothrow) FlucTtmlBlendMulti ();
  if (!m)
    return FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY;
  for (int d : devs) {
    FlucTtmlBlend *t = nullptr;
    const int rc = d < 0 ? FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT : fluc_ttmlblend_new (d, &t);
    if (rc) {
      fluc_ttmlblend_multi_free (m);
      return rc;
    }
    m->ctx.push_back (t);
    m->device.push_back (d);
  }
  *out = m;
  return 0;
}

void
fluc_ttmlblend_multi_free (FlucTtmlBlendMulti *thiz)
{
  if (!thiz)
    return;
  for (FlucTtmlBlend *t : thiz->ctx)
    fluc_ttmlblend_free (t);
  delete thiz;
}

uint32_t
fluc_ttmlblend_multi_size (FlucTtmlBlendMulti *thiz)
{
  return thiz ? (uint32_t) thiz->ctx.size () : 0u;
}

FlucTtmlBlend *
fluc_ttmlblend_multi_context (FlucTtmlBlendMulti *thiz, uint32_t stream)
{
  return thiz && !thiz->ctx.empty () ? thiz->ctx[stream % thiz->ctx.size ()] : nullptr;
}

int
fluc_ttmlblend_multi_device (FlucTtmlBlendMulti *thiz, uint32_t stream)
{
  return thiz && !thiz->ctx.empty () ? thiz->device[stream % thiz->ctx.size ()] : -1;
}

int
fluc_ttmlblend_multi_sync (FlucTtmlBlendMulti *thiz)
{
  if (!thiz)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  int ret = 0;
  /* launch everywhere first, then wait: the devices work at the same time */
  for (FlucTtmlBlend *t : thiz->ctx) {
    const int rc = fluc_ttmlblend_flush (t);
    ret = ret ? ret : rc;
  }
  for (FlucTtmlBlend *t : thiz->ctx) {
    const int rc = fluc_ttmlblend_sync (t);
    ret = ret ? ret : rc;
  }
  return ret;
}

void
fluc_ttmlblend_multi_stats_copy (FlucTtmlBlendMulti *thiz, FlucTtmlBlendStats *out)
{
  if (!thiz || !out)
    return;
  FlucTtmlBlendStats sum = {};
  for (FlucTtmlBlend *t : thiz->ctx) {
    FlucTtmlBlendStats s = {};
    fluc_ttmlblend_stats_copy (t, &s);
    sum.frames_blended += s.frames_blended;
    sum.launches += s.launches;
    sum.group_launches += s.group_launches;
    sum.prepare_launches += s.prepare_launches;
    sum.overlays_set += s.overlays_set;
    sum.algorithmic_bytes += s.algorithmic_bytes;
    sum.h2d_bytes += s.h2d_bytes;
    sum.d2h_bytes += s.d2h_bytes;
    sum.kernel_ms += s.kernel_ms;
    sum.kernel_ms_launches += s.kernel_ms_launches;
    sum.cache_bytes += s.cache_bytes;
    sum.multi_launches += s.multi_launches;
    sum.lazy_launches += s.lazy_launches;
    sum.dependent_launches += s.dependent_launches;
    sum.overlays_updated += s.overlays_updated;
    sum.staged_frames += s.staged_frames;
    sum.opaque_skip_launches += s.opaque_skip_launches;
    sum.host_dma_batches += s.host_dma_batches;
  }
  *out = sum;
}

/* ---- observability --------------------------------------------------- */

void
fluc_ttmlblend_stats_copy (FlucTtmlBlend *thiz, FlucTtmlBlendStats *out)
{
  if (!thiz || !out)
    return;
  std::unique_lock<std::mutex> lk (thiz->c.mu);
  cudaSetDevice (thiz->c.device);
  reap_batches (&thiz->c);
  *out = thiz->c.stats;
  /* what the overlay caches hold: everything they allocate is stream-ordered pool memory */
  uint64_t used = 0;
  if (cudaMemPoolGetAttribute (thiz->c.mem_pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess)
    out->cache_bytes = used;
  else
    cudaGetLastError ();
}

void
fluc_ttmlblend_stats_reset (FlucTtmlBlend *thiz)
{
  if (!thiz)
    return;
  std::unique_lock<std::mutex> lk (thiz->c.mu);
  cudaSetDevice (thiz->c.device);
  reap_batches (&thiz->c);
  thiz->c.stats = FlucTtmlBlendStats ();
}

int
fluc_ttmlblend_set_profiling (FlucTtmlBlend *thiz, int enabled)
{
  ENTER (thiz);
  c->profiling = enabled != 0;
  if (enabled > 0)
    c->profile_every = (uint32_t) enabled;
  c->profile_seq = 0;
  return 0;
}

int
fluc_ttmlblend_timer_begin (FlucTtmlBlend *thiz)
{
  ENTER (thiz);
  int rc = launch_pending (c);
  if (rc)
    return rc;
  CU (c, cudaEventRecord (c->timer0, c->blend_stream));
  return 0;
}

int
fluc_ttmlblend_timer_end (FlucTtmlBlend *thiz, double *ms)
{
  ENTER (thiz);
  int rc = launch_pending (c);
  if (rc)
    return rc;
  CU (c, cudaEventRecord (c->timer1, c->blend_stream));
  CU (c, cudaEventSynchronize (c->timer1));
  float f = 0.f;
  CU (c, cudaEventElapsedTime (&f, c->timer0, c->timer1));
  if (ms)
    *ms = f;
  reap_batches (c);
  return 0;
}

int
fluc_ttmlblend_scrub_l2 (FlucTtmlBlend *thiz, size_t bytes)
{
  ENTER (thiz);
  if (bytes > c->scrub_bytes) {
    if (c->scrub)
      CU (c, cudaFree (c->scrub));
    c->scrub = nullptr;
    c->scrub_bytes = 0;
    CU (c, cudaMalloc ((void **) &c->scrub, bytes));
    c->scrub_bytes = bytes;
  }
  CU (c, launch_scrub (c->scrub, bytes, c->blend_stream));
  return 0;
}

int
fluc_ttmlblend_pcie_probe (FlucTtmlBlend *thiz, int mode, size_t bytes, double seconds, double *gbs)
{
  ENTER (thiz);
  if (mode < 0 || mode > 1 || bytes < 4096 || bytes > ((size_t) 1 << 31) || !(seconds > 0.0) || seconds > 10.0)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  bytes &= ~(size_t) 4095;
  int rc = launch_pending (c);
  if (rc)
    return rc;
  /* buffers of its own, nothing shared with frames in flight; the context stays unlocked while
   * the probe runs (it touches only these buffers and the two copy streams of host DMA batches,
   * drained first) */
  uint8_t *h_in = nullptr, *h_out = nullptr, *d_in = nullptr, *d_out = nullptr;
  auto cleanup = [&]() {
    if (h_in) cudaFreeHost (h_in);
    if (h_out) cudaFreeHost (h_out);
    if (d_in) cudaFree (d_in);
    if (d_out) cudaFree (d_out);
  };
  {
    NumaScope numa (c);
    if (cudaHostAlloc ((void **) &h_in, bytes, cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc ((void **) &h_out, bytes, cudaHostAllocDefault) != cudaSuccess ||
        cudaMalloc ((void **) &d_in, bytes) != cudaSuccess || cudaMalloc ((void **) &d_out, bytes) != cudaSuccess) {
      cudaGetLastError ();
      cleanup ();
      return FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY;
    }
  }
  memset (h_in, 0x5a, bytes);
  memset (h_out, 0xa5, bytes);
  cudaStream_t s1 = c->dma_in, s2 = c->dma_out;
  cudaStreamSynchronize (s1);
  cudaStreamSynchronize (s2);
  lk.unlock ();
  auto issue = [&]() -> cudaError_t {
    if (mode == 0) {
      cudaError_t e = cudaMemcpyAsync (d_in, h_in, bytes, cudaMemcpyHostToDevice, s1);
      if (e != cudaSuccess)
        return e;
      return cudaMemcpyAsync (h_out, d_out, bytes, cudaMemcpyDeviceToHost, s2);
    }
    return launch_pcie_probe (h_in, bytes, s1);
  };
  cudaError_t e = issue ();
  if (e == cudaSuccess) e = cudaStreamSynchronize (s1);
  if (e == cudaSuccess) e = cudaStreamSynchronize (s2);
  const auto t0 = std::chrono::steady_clock::now ();
  double t = 0.0;
  uint64_t iters = 0;
  while (e == cudaSuccess && t < seconds) {
    e = issue ();
    if (e == cudaSuccess) e = issue ();
    if (e == cudaSuccess) e = cudaStreamSynchronize (s1);
    if (e == cudaSuccess) e = cudaStreamSynchronize (s2);
    iters += 2;
    t = std::chrono::duration<double> (std::chrono::steady_clock::now () - t0).count ();
  }
  lk.lock ();
  cleanup ();
  if (e != cudaSuccess) {
    c->cuda_error = std::string ("pcie_probe: ") + cudaGetErrorString (e);
    c->sticky = FLUC_TTMLBLEND_ERROR_CUDA;
    return c->sticky;
  }
  if (gbs)
    *gbs = (double) bytes * (double) iters / t / 1e9;
  return 0;
}

void *
fluc_ttmlblend_stream_handle (FlucTtmlBlend *thiz)
{
  return thiz ? (void *) thiz->c.blend_stream : nullptr;
}

}  /* extern "C" */
