/*
 * overlay_cache.cu -- the per-stream overlay cache: upload of the cue rectangles, auto-crop to
 * non-transparent row runs, the once-per-cue prepare launches, and stream-ordered deferred frees.
 * Producer side in the reference: gst_ttmlrender_gen_buffer,
 * /root/reference/plugins/ttml/gstttmlrender.c:1427-1478.
 */
#include "ttmlblend_internal.h"

#include <numeric>

namespace tbh {

/* Frees device memory once everything already queued on any of the
 * context's streams has run: the reaper stream waits for a fence event on
 * each of them, then frees in stream order. */
void
free_deferred (Ctx *c, const std::vector<void *> &ptrs)
{
  if (ptrs.empty ())
    return;
  const cudaStream_t all[2] = { c->blend_stream, c->up_stream };
  for (int i = 0; i < 2; i++) {
    if (!all[i])
      continue;
    cudaEventRecord (c->ev_fence[i], all[i]);
    cudaStreamWaitEvent (c->reaper, c->ev_fence[i], 0);
  }
  for (void *p : ptrs)
    cudaFreeAsync (p, c->reaper);
}

DevBlock::~DevBlock ()
{
  if (ctx && ptr)
    free_deferred (ctx, { ptr });
}

/* Blocks nobody else holds are freed in one go (one fence per stream instead of one per block);
 * blocks a newer overlay of the stream shares (overlay_update) live on with it. */
Overlay::~Overlay ()
{
  std::vector<void *> ptrs;
  auto take = [&ptrs](std::shared_ptr<DevBlock> &b) {
    if (b && b.use_count () == 1 && b->ptr) {
      ptrs.push_back (b->ptr);
      b->ptr = nullptr;
    }
  };
  for (RawRect &r : rects)
    take (r.block);
  for (OverlayBox &b : boxes)
    take (b.src.block);
  for (auto &p : prepared) {
    for (PreparedRect &pr : p->per_rect) {
      for (auto &b : pr.blocks)
        take (b);
      for (auto &b : pr.avg_blocks)
        take (b);
    }
    take (p->table_block);
  }
  if (ctx)
    free_deferred (ctx, ptrs);
}

Prepared::~Prepared ()
{
  if (ready)
    cudaEventDestroy (ready);
}

/* ---------------------------------------------------------------------- */
/* prepare: raw BGRA rectangle -> per-plane prepared overlay              */

static std::shared_ptr<DevBlock>
make_block (Ctx *c, void *ptr)
{
  std::shared_ptr<DevBlock> b (new DevBlock ());
  b->ctx = c;
  b->ptr = ptr;
  return b;
}

/* a stream-ordered allocation on the upload stream */
static int
dev_block (Ctx *c, size_t bytes, std::shared_ptr<DevBlock> *out)
{
  void *ptr = nullptr;
  CU (c, cudaMallocFromPoolAsync (&ptr, std::max<size_t> (bytes, 16), c->mem_pool, c->up_stream));
  *out = make_block (c, ptr);
  return 0;
}

static int
dev_alloc (Ctx *c, std::vector<std::shared_ptr<DevBlock>> *blocks, size_t bytes, uint8_t **out)
{
  std::shared_ptr<DevBlock> b;
  int rc = dev_block (c, bytes, &b);
  if (rc)
    return rc;
  *out = static_cast<uint8_t *> (b->ptr);
  blocks->push_back (std::move (b));
  return 0;
}

/* One prepare launch of n_elems elements per row, counted -- or, with a batch (a move,
 * overlay_set_positions), one item of its single launch. Averaged chroma keeps its own kernel. */
static int
issue_prepare (Ctx *c, const PrepareParams &pp, int n_elems, std::vector<PrepareItem> *batch)
{
  if (batch && !pp.chroma_average) {
    if (n_elems > 0 && pp.rows > 0)
      batch->push_back ({ pp, n_elems, 0 });
    return 0;
  }
  CU (c, launch_prepare (pp, n_elems, c->up_stream));
  c->stats.prepare_launches++;
  return 0;
}

/* The prepare parameters every plane of a rectangle shares; false when nothing of it is inside
 * the frame. */
static bool
rect_params (const RawRect &rr, int format, int W, int H, PrepareParams &pp)
{
  /* gst_video_blend clipping at all four edges (a rectangle of the composition form keeps the
   * part above / left of the frame on the device, raw pixel (0,0) at frame (rr.x, rr.y)) */
  const int cx0 = std::max (rr.x, 0), cy0 = std::max (rr.y, 0);
  const int cx1 = std::min (rr.x + rr.w, W), cy1 = std::min (rr.y + rr.h, H);
  if (cx1 <= cx0 || cy1 <= cy0)
    return false;
  pp = {};
  pp.raw = rr.dev;
  pp.raw_pitch = rr.pitch;
  pp.raw_w = rr.w;
  pp.raw_h = rr.h;
  pp.fx = rr.x;
  pp.fy = rr.y;
  pp.cx0 = cx0; pp.cy0 = cy0; pp.cx1 = cx1; pp.cy1 = cy1;
  pp.ga = rr.ga;
  pp.premul = rr.premul ? 1 : 0;
  pp.sub_x = format_sub_x (format);
  pp.sub_y = format_sub_y (format);
  return true;
}

/* One plane group of a rectangle: n_planes planes (alpha first) over the byte columns [b0, b1)
 * of a destination plane, widened to whole 16-byte vectors, and its rows [y0, y1), prepared in
 * `mode` with elem_bytes bytes per kernel element. Their blocks go to `blocks`. `ref` gets the
 * span, ga 255 and the first two planes; `planes` all of them. */
static int
prepare_planes (Ctx *c, PrepareParams &pp, int mode, int b0, int b1, int y0, int y1, int n_planes, int elem_bytes,
    std::vector<std::shared_ptr<DevBlock>> *blocks, std::vector<PrepareItem> *batch, RectRef &ref, uint8_t *planes[3])
{
  ref = {};
  ref.v0 = b0 / 16;
  ref.v1 = ceil_div (b1, 16);
  ref.y0 = y0;
  ref.y1 = y1;
  ref.pitch = (ref.v1 - ref.v0) * 16;
  ref.ga = 255;
  const size_t bytes = (size_t) ref.pitch * (y1 - y0);
  for (int k = 0; k < 3; k++)
    planes[k] = nullptr;
  for (int k = 0; k < n_planes; k++) {
    const int rc = dev_alloc (c, blocks, bytes, &planes[k]);
    if (rc)
      return rc;
  }
  ref.a = planes[0];
  ref.c = planes[1];
  pp.mode = mode;
  pp.out_a = planes[0]; pp.out_c = planes[1]; pp.out_c2 = planes[2];
  pp.out_pitch = ref.pitch;
  pp.v0 = ref.v0;
  pp.row0 = y0;
  pp.rows = y1 - y0;
  return issue_prepare (c, pp, ref.pitch / elem_bytes, batch);
}

/* The chroma planes of a planar / semi-planar YUV format: the samples sited on the even pixel
 * of each pair / the even line of each line pair, as far as the format subsamples (parity);
 * with the non-parity 2x2 average of 4:2:0 (avg) every sample with at least one covered pixel.
 * Nothing for the one-plane formats. Their planes go to `blocks`. */
static int
prepare_chroma (Ctx *c, PrepareParams pp, int format, bool avg, std::vector<std::shared_ptr<DevBlock>> *blocks,
    PreparedRect &out, std::vector<PrepareItem> *batch)
{
  const int n_planes = format_planes (format);
  const int sx = pp.sub_x, sy = pp.sub_y;
  pp.chroma_average = avg ? 1 : 0;
  const int bx0 = avg ? pp.cx0 / 2 : ceil_div (pp.cx0, sx), bx1 = ceil_div (pp.cx1, sx);
  const int by0 = avg ? pp.cy0 / 2 : ceil_div (pp.cy0, sy), by1 = ceil_div (pp.cy1, sy);
  if (n_planes < 2 || bx1 <= bx0 || by1 <= by0)
    return 0;
  RectRef ref;
  uint8_t *planes[3];
  int rc;
  if (n_planes == 3) {
    /* alpha, U, V: one byte per sample */
    if ((rc = prepare_planes (c, pp, PM_CHROMA_PLANAR, bx0, bx1, by0, by1, 3, 1, blocks, batch, ref, planes)))
      return rc;
    const int pu = format == FLUC_TTMLBLEND_FORMAT_YV12 ? 2 : 1;
    out.refs[out.n_refs++] = { pu, ref };
    ref.c = planes[2];
    out.refs[out.n_refs++] = { 3 - pu, ref };
  } else {
    /* alpha pairs and interleaved U,V: two bytes per sample */
    const int mode = (format == FLUC_TTMLBLEND_FORMAT_NV21 || format == FLUC_TTMLBLEND_FORMAT_NV61) ?
        PM_CHROMA_VU : PM_CHROMA_UV;
    if ((rc = prepare_planes (c, pp, mode, 2 * bx0, 2 * bx1, by0, by1, 2, 2, blocks, batch, ref, planes)))
      return rc;
    out.refs[out.n_refs++] = { 1, ref };
  }
  return 0;
}

/* Averaged 4:2:0 chroma at the box's global alpha `ga`: asrc = a*ga/255 per pixel before the
 * 2x2 sums (BLENDSPEC section 7), so unlike every other PLANE8 plane the value is folded in
 * here and the blend leaves these refs alone. Nothing at 0: the box is not blended. */
static int
prepare_avg_chroma (Ctx *c, PrepareParams pp, int format, int ga, PreparedRect &out)
{
  out.avg_ga = ga;
  if (ga == 0)
    return 0;
  pp.ga = ga;
  return prepare_chroma (c, pp, format, true, &out.avg_blocks, out, nullptr);
}

/* the prepare mode of a format's first plane group: luma, the packed 4:2:2 / 3-byte 4:4:4
 * bytes, or the pixel words */
static int
first_mode (int format)
{
  switch (format) {
    case FLUC_TTMLBLEND_FORMAT_YUY2: return PM_YUY2;
    case FLUC_TTMLBLEND_FORMAT_UYVY: return PM_UYVY;
    case FLUC_TTMLBLEND_FORMAT_YVYU: return PM_YVYU;
    case FLUC_TTMLBLEND_FORMAT_VYUY: return PM_VYUY;
    case FLUC_TTMLBLEND_FORMAT_v308: return PM_V308;
    case FLUC_TTMLBLEND_FORMAT_IYU2: return PM_IYU2;
    case FLUC_TTMLBLEND_FORMAT_RGB: return PM_RGB24;
    case FLUC_TTMLBLEND_FORMAT_BGR: return PM_BGR24;
    case FLUC_TTMLBLEND_FORMAT_AYUV: return PM_PACKED_AYUV;
    case FLUC_TTMLBLEND_FORMAT_ARGB: return PM_PACKED_ARGB;
    case FLUC_TTMLBLEND_FORMAT_ABGR: return PM_PACKED_ABGR;
    case FLUC_TTMLBLEND_FORMAT_RGBA: return PM_PACKED_RGBA;
    case FLUC_TTMLBLEND_FORMAT_BGRA: return PM_PACKED_BGRA;
    default: return PM_LUMA;
  }
}

/* Prepares one rectangle for one destination format: allocates its planes, runs the prepare
 * kernel(s) on the upload stream (or adds them to `batch`, issue_prepare), and notes how each
 * destination plane sees it. ga_now is the current global alpha of its box, which only averaged
 * chroma folds in. */
static int
prepare_rect (Ctx *c, const RawRect &rr, int format, int W, int H, bool chroma_average, int ga_now,
    PreparedRect &out, std::vector<PrepareItem> *batch)
{
  const int kind = plane_kind (format);
  PrepareParams pp;
  if (!rect_params (rr, format, W, H, pp))
    return 0;
  if (rr.ga == 0)
    return 0;                 /* asrc == 0 everywhere: blends nothing */
  const int cx0 = pp.cx0, cx1 = pp.cx1;
  /* the first plane group's byte columns: a luma plane (byte == pixel), alpha + colour planes */
  int b0 = cx0, b1 = cx1, n_planes = 2, elem_bytes = 1;
  if (format_packed_422 (format)) {
    /* YUY2 / UYVY: one plane of macropixels, every byte gets its own alpha + colour */
    b0 = 4 * (cx0 / 2);
    b1 = 4 * ceil_div (cx1, 2);
    elem_bytes = 4;
  } else if (kind == PK_PLANE8_RGB || format_packed_444_3 (format)) {
    /* v308 / IYU2 / RGB / BGR: one plane, three bytes per pixel, every byte its own alpha + colour */
    b0 = 3 * cx0;
    b1 = 3 * cx1;
  } else if (kind != PK_PLANE8) {
    /* one plane of pixel words */
    b0 = 4 * cx0;
    b1 = 4 * cx1;
    n_planes = 1;
    elem_bytes = 4;
  }
  RectRef ref;
  uint8_t *planes[3];
  const int rc = prepare_planes (c, pp, first_mode (format), b0, b1, pp.cy0, pp.cy1, n_planes, elem_bytes,
      &out.blocks, batch, ref, planes);
  if (rc)
    return rc;
  if (kind != PK_PLANE8) {
    /* the RGB pair and the pixel words keep the source colours and the rectangle's flags for the
     * blend (AYUV's colours are converted, so premultiplied ones are not) */
    ref.ga = rr.ga;
    ref.src_premul = (format != FLUC_TTMLBLEND_FORMAT_AYUV && rr.premul) ? 1 : 0;
  }
  out.refs[out.n_refs++] = { 0, ref };
  if (chroma_average && pp.sub_x == 2 && pp.sub_y == 2)
    return prepare_avg_chroma (c, pp, format, ga_now, out);
  return prepare_chroma (c, pp, format, false, &out.blocks, out, batch);
}

/* the PLANE8 kinds fold a rectangle's global alpha into its prepared alpha bytes; the packed kinds
 * give it to the blend */
static bool
folds_ga (int format)
{
  const int kind = plane_kind (format);
  return kind == PK_PLANE8 || kind == PK_PLANE8_RGB;
}

/* The rectangle tables of P with every box's current global alpha: a box at 0 drops out (no
 * band, no window in place), the others give it to the blend where the prepare did not fold it
 * in -- RectRef::ga for the Cs*ga terms, RectRef::a_ga for the alpha bytes of the PLANE8 kinds.
 * Averaged 4:2:0 chroma has it folded in (prepare_avg_chroma). A move's batch of prepares
 * (overlay_set_positions) goes out here as one launch; when its items do not fit in the kernel
 * parameters they are uploaded in the tables' allocation, behind them. */
static int
prepare_assemble (Ctx *c, Prepared *P, const Overlay *ov, std::vector<PrepareItem> *batch)
{
  for (int pl = 0; pl < 3; pl++)
    P->h_rects[pl].clear ();
  const int kind = plane_kind (P->format);
  const bool planes = folds_ga (P->format);
  P->fade = false;
  for (const OverlayBox &b : ov->boxes)
    for (uint32_t i = b.first_rect; i < b.first_rect + b.n_rects; i++) {
      const PreparedRect &pr = P->per_rect[i];
      if (b.ga == 0)
        continue;
      const bool folded = planes && ov->rects[i].ga != 255;
      for (int k = 0; k < pr.n_refs; k++) {
        RectRef ref = pr.refs[k].ref;
        ref.a_ga = 255;
        if (!folded && !(pr.avg_ga >= 0 && pr.refs[k].plane != 0)) {
          if (kind != PK_PLANE8)
            ref.ga = b.ga;
          if (planes)
            ref.a_ga = b.ga;
        }
        P->fade = P->fade || ref.a_ga != 255;
        P->h_rects[pr.refs[k].plane].push_back (ref);
      }
    }
  /* rectangle tables: one contiguous device array, plane after plane */
  {
    size_t total = 0;
    for (int pl = 0; pl < 3; pl++) {
      if (P->h_rects[pl].size () > FLUC_TTMLBLEND_MAX_RECTANGLES)
        return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
      P->rect_off[pl] = (int32_t) total;
      total += P->h_rects[pl].size ();
    }
    const uint32_t n_items = batch ? (uint32_t) batch->size () : 0;
    const uint32_t ctas = n_items ? prepare_batch_plan (batch->data (), n_items) : 0;
    const size_t item_bytes = n_items > kPrepareBatchInline ? n_items * sizeof (PrepareItem) : 0;
    if (total || item_bytes) {
      int rc;
      if ((rc = dev_block (c, total * sizeof (RectRef) + item_bytes, &P->table_block)))
        return rc;
    }
    if (n_items) {
      const PrepareItem *d_items = nullptr;
      if (item_bytes) {
        P->h_items = std::move (*batch);      /* the async copy's source lives as long as P */
        d_items = reinterpret_cast<const PrepareItem *> (static_cast<uint8_t *> (P->table_block->ptr) +
            total * sizeof (RectRef));
        CU (c, cudaMemcpyAsync ((void *) d_items, P->h_items.data (), item_bytes, cudaMemcpyHostToDevice,
                c->up_stream));
      }
      CU (c, launch_prepare_batch (item_bytes ? P->h_items.data () : batch->data (), n_items, d_items, ctas,
              c->up_stream));
      c->stats.prepare_launches++;
    }
    if (total) {
      P->h_rects_all.clear ();
      for (int pl = 0; pl < 3; pl++)
        P->h_rects_all.insert (P->h_rects_all.end (), P->h_rects[pl].begin (), P->h_rects[pl].end ());
      uint8_t *d = static_cast<uint8_t *> (P->table_block->ptr);
      /* h_rects_all lives as long as the Prepared: safe source for the async copy */
      CU (c, cudaMemcpyAsync (d, P->h_rects_all.data (), total * sizeof (RectRef),
              cudaMemcpyHostToDevice, c->up_stream));
      P->d_rects_all = reinterpret_cast<RectRef *> (d);
      for (int pl = 0; pl < 3; pl++)
        if (!P->h_rects[pl].empty ())
          P->d_rects[pl] = P->d_rects_all + P->rect_off[pl];
    }
  }
  CU (c, cudaEventCreateWithFlags (&P->ready, cudaEventDisableTiming));
  CU (c, cudaEventRecord (P->ready, c->up_stream));
  return 0;
}

/* the current global alpha of the box that rectangle i of ov belongs to */
static int
box_ga (const Overlay *ov, size_t i)
{
  for (const OverlayBox &b : ov->boxes)
    if (i >= b.first_rect && i < b.first_rect + b.n_rects)
      return b.ga;
  return ov->rects[i].ga;
}

/* the pixels of ov's rectangles as handed in, clipped to a W x H frame (algorithmic bytes) */
static uint64_t
declared_px (const Overlay *ov, int W, int H)
{
  uint64_t px = 0;
  for (const FlucTtmlBlendRect &d : ov->declared) {
    const int w = std::min (d.x + d.w, W) - std::max (d.x, 0), h = std::min (d.y + d.h, H) - std::max (d.y, 0);
    if (w > 0 && h > 0)
      px += (uint64_t) w * (uint64_t) h;
  }
  return px;
}

/* Can rectangle `now` use the planes prepared from `was`: equal in everything rect_params and
 * prepare_rect read. The global alpha counts where the prepare folds it in (folds_ga); for the
 * packed kinds only whether it is 0 (nothing prepared). */
static bool
same_prepare (const RawRect &now, const RawRect &was, bool folded)
{
  return now.dev == was.dev && now.pitch == was.pitch && now.w == was.w && now.h == was.h && now.x == was.x &&
      now.y == was.y && now.premul == was.premul && (folded ? now.ga == was.ga : (now.ga == 0) == (was.ga == 0));
}

/* Builds the Prepared of nv for (format, W, H, chroma_average) and adds it to nv->prepared. For a
 * new generation of an overlay (overlay_update, a fade, a move), `old` is the Prepared of the
 * previous generation `prev` for the same four, and from_old[i] the rectangle of prev that
 * rectangle i of nv comes from (-1: none). A rectangle keeps the planes of the one it comes from when the two
 * are the same for the prepare (same_prepare), and its averaged chroma as well when that was
 * prepared at its box's current global alpha; otherwise only the averaged chroma is prepared again
 * at the new value. Every other rectangle is prepared from its raw pixels: with `batched`
 * (overlay_set_positions) in one batch launch. */
static int
build_prepared (Ctx *c, Overlay *nv, int format, int W, int H, bool chroma_average, const Overlay *prev = nullptr,
    const Prepared *old = nullptr, const std::vector<int> *from_old = nullptr, bool batched = false)
{
  std::unique_ptr<Prepared> P (new Prepared ());
  P->format = format;
  P->W = W;
  P->H = H;
  P->chroma_average = chroma_average;
  P->overlay_px = declared_px (nv, W, H);
  P->used = old ? old->used : false;
  P->per_rect.resize (nv->rects.size ());
  const bool folded = folds_ga (format);
  std::vector<PrepareItem> items;
  std::vector<PrepareItem> *batch = batched ? &items : nullptr;
  for (size_t i = 0; i < nv->rects.size (); i++) {
    const RawRect &rr = nv->rects[i];
    const int j = old ? (*from_old)[i] : -1;
    const PreparedRect *was = j >= 0 ? &old->per_rect[(size_t) j] : nullptr;
    const int ga = box_ga (nv, i);
    PreparedRect &pr = P->per_rect[i];
    PrepareParams pp;
    int rc = 0;
    if (!was || !same_prepare (rr, prev->rects[(size_t) j], folded)) {
      rc = prepare_rect (c, rr, format, W, H, chroma_average, ga, pr, batch);
    } else if (was->avg_ga >= 0 && was->avg_ga != ga && rect_params (rr, format, W, H, pp)) {
      /* the luma planes as they were, the averaged chroma at the new value */
      pr.blocks = was->blocks;
      for (int k = 0; k < was->n_refs; k++)
        if (was->refs[k].plane == 0)
          pr.refs[pr.n_refs++] = was->refs[k];
      rc = prepare_avg_chroma (c, pp, format, ga, pr);
    } else {
      pr = *was;
    }
    if (rc)
      return rc;
  }
  const int rc = prepare_assemble (c, P.get (), nv, batch);
  if (rc)
    return rc;
  nv->prepared.push_back (std::move (P));
  return 0;
}

int
prepare_overlay (Ctx *c, Overlay *ov, int format, int W, int H, Prepared **out)
{
  for (auto &p : ov->prepared)
    if (p->format == format && p->W == W && p->H == H && p->chroma_average == c->chroma_average) {
      *out = p.get ();
      return 0;
    }

  NvtxRange nvtx ("ttmlblend.prepare_overlay");
  TBLOG (2, "prepare overlay: format %d, %dx%d, %zu rectangle(s)", format, W, H, ov->rects.size ());
  /* a half-built one (out of memory, too many rectangles) goes back with its blocks */
  const int rc = build_prepared (c, ov, format, W, H, c->chroma_average);
  if (rc)
    return rc;
  *out = ov->prepared.back ().get ();
  return 0;
}


/* ---------------------------------------------------------------------- */
/* plane jobs                                                             */

/* Decomposes possibly overlapping region rectangles into disjoint ones that
 * cover the same pixels, so that every pixel of the ttmlrender image is
 * blended exactly once. */
std::vector<FlucTtmlBlendRect>
disjoint_cover (const std::vector<FlucTtmlBlendRect> &in)
{
  std::vector<int> ys;
  for (auto &r : in) {
    ys.push_back (r.y);
    ys.push_back (r.y + r.h);
  }
  std::sort (ys.begin (), ys.end ());
  ys.erase (std::unique (ys.begin (), ys.end ()), ys.end ());
  std::vector<FlucTtmlBlendRect> out;
  for (size_t i = 0; i + 1 < ys.size (); i++) {
    const int y0 = ys[i], y1 = ys[i + 1];
    std::vector<std::pair<int, int>> xs;
    for (auto &r : in)
      if (r.y <= y0 && r.y + r.h >= y1)
        xs.push_back ({ r.x, r.x + r.w });
    std::sort (xs.begin (), xs.end ());
    std::vector<std::pair<int, int>> merged;
    for (auto &x : xs) {
      if (!merged.empty () && x.first <= merged.back ().second)
        merged.back ().second = std::max (merged.back ().second, x.second);
      else
        merged.push_back (x);
    }
    for (auto &m : merged) {
      bool grown = false;
      for (auto &o : out)
        if (o.x == m.first && o.w == m.second - m.first && o.y + o.h == y0) {
          o.h += y1 - y0;
          grown = true;
          break;
        }
      if (!grown)
        out.push_back ({ m.first, y0, m.second - m.first, y1 - y0 });
    }
  }
  return out;
}

/* Cuts a rectangle down to where it is not transparent: runs of non-empty
 * rows (text lines, boxes) become separate sub-rectangles, each as wide as its
 * outermost non-transparent pixels. Pixels with alpha 0 never change the frame
 * (BLENDSPEC section 2, `continue`), so dropping them is exact; what it buys is
 * that ttmlrender's frame-sized, mostly empty image costs overlay reads, ALU
 * work and -- for host frames -- PCIe traffic only where there is a cue. */
void
crop_runs (const std::vector<int2> &spans, int min_gap, size_t max_runs, std::vector<FlucTtmlBlendRect> &out)
{
  struct Run { int y0, y1, x0, x1; };
  std::vector<Run> runs;
  for (int y = 0; y < (int) spans.size (); y++) {
    if (spans[y].y < spans[y].x)
      continue;
    if (!runs.empty () && y - runs.back ().y1 < min_gap) {
      Run &r = runs.back ();
      r.y1 = y + 1;
      r.x0 = std::min (r.x0, spans[y].x);
      r.x1 = std::max (r.x1, spans[y].y + 1);
    } else {
      runs.push_back ({ y, y + 1, spans[y].x, spans[y].y + 1 });
    }
  }
  while (runs.size () > max_runs) {
    size_t best = 0;
    for (size_t i = 1; i + 1 < runs.size (); i++)
      if (runs[i + 1].y0 - runs[i].y1 < runs[best + 1].y0 - runs[best].y1)
        best = i;
    runs[best].y1 = runs[best + 1].y1;
    runs[best].x0 = std::min (runs[best].x0, runs[best + 1].x0);
    runs[best].x1 = std::max (runs[best].x1, runs[best + 1].x1);
    runs.erase (runs.begin () + best + 1);
  }
  for (const Run &r : runs)
    out.push_back ({ r.x0, r.y0, r.x1 - r.x0, r.y1 - r.y0 });
}

/* A rectangle whose pixels already sit in device memory, on its way into an overlay. */
struct Up {
  RawRect rr;
  std::vector<int2> spans;
  std::vector<int> groups;      /* per row: 16-pixel groups with any alpha */
  std::vector<int> raw;         /* both as they come back from the GPU in one copy: h x int2, then h x int */
  uint32_t slot = 0;            /* OverlayBox::slot */
  BoxSource src;                /* OverlayBox::src */
};

/* Is this pointer device memory (a cue produced on the GPU, or left there by a previous stage)? */
static bool
on_device (const void *p)
{
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes (&attr, p) != cudaSuccess) {
    cudaGetLastError ();
    return false;
  }
  return attr.type == cudaMemoryTypeDevice;
}

/* What an install does to the context's counters, added once the lock is held again. */
struct InstallStats {
  uint64_t h2d_bytes = 0;
  uint32_t launches = 0;
};

/* CU for the parts of an install that run without the context lock: the lock is taken back
 * before the error is recorded and reported. */
#define CUU(ctx, lk, call) do {                                              \
    cudaError_t eu_ = (call);                                                \
    if (eu_ != cudaSuccess) {                                                \
      if (!(lk).owns_lock ())                                                \
        (lk).lock ();                                                        \
      (ctx)->cuda_error = std::string (#call) + ": " + cudaGetErrorString (eu_); \
      if (eu_ == cudaErrorMemoryAllocation) {                                \
        cudaGetLastError ();                                                 \
        return FLUC_TTMLBLEND_ERROR_OUT_OF_MEMORY;                           \
      }                                                                      \
      (ctx)->sticky = FLUC_TTMLBLEND_ERROR_CUDA;                             \
      return FLUC_TTMLBLEND_ERROR_CUDA;                                      \
    }                                                                        \
  } while (0)

/* Queues the row-span scan of one device-resident rectangle on the upload stream. */
static int
scan_rows (Ctx *c, std::unique_lock<std::mutex> &lk, Up &u)
{
  if (!c->autocrop)
    return 0;
  void *sp = nullptr;
  const size_t nb = (size_t) u.rr.h * (sizeof (int2) + sizeof (int));
  CUU (c, lk, cudaMallocFromPoolAsync (&sp, nb, c->mem_pool, c->up_stream));
  u.raw.resize ((size_t) u.rr.h * 3);
  int2 *d_spans = static_cast<int2 *> (sp);
  int *d_groups = reinterpret_cast<int *> (d_spans + u.rr.h);
  CUU (c, lk, launch_rowspan (u.rr.dev, u.rr.pitch, u.rr.w, u.rr.h, d_spans, d_groups, c->up_stream));
  CUU (c, lk, cudaMemcpyAsync (u.raw.data (), sp, nb, cudaMemcpyDeviceToHost, c->up_stream));   /* one copy for both */
  CUU (c, lk, cudaFreeAsync (sp, c->up_stream));
  return 0;
}

/* Queues the upload of rr.w x rr.h BGRA pixels from `src` into a block of rr's own on the upload
 * stream. cudaMemcpyDefault: the pixels may just as well be in device memory already (UVA tells);
 * host pixels count into st.h2d_bytes. */
static int
upload_rect (Ctx *c, std::unique_lock<std::mutex> &lk, const uint8_t *src, int stride, RawRect &rr, InstallStats &st)
{
  rr.pitch = (int) align_up ((size_t) rr.w * 4, 256);
  void *d = nullptr;
  CUU (c, lk, cudaMallocFromPoolAsync (&d, (size_t) rr.pitch * rr.h, c->mem_pool, c->up_stream));
  rr.block = make_block (c, d);
  rr.dev = static_cast<uint8_t *> (d);
  CUU (c, lk, cudaMemcpy2DAsync (rr.dev, rr.pitch, src, stride, (size_t) rr.w * 4, rr.h, cudaMemcpyDefault,
          c->up_stream));
  if (!on_device (src))
    st.h2d_bytes += (uint64_t) rr.w * 4 * rr.h;
  return 0;
}

/* Waits for what the install queued on the upload stream while unlocked -- the caller's pixels
 * must be consumed and the row spans back before it returns -- and takes the context lock back. */
static int
wait_uploads (Ctx *c, std::unique_lock<std::mutex> &lk)
{
  CUU (c, lk, cudaStreamSynchronize (c->up_stream));
  if (!lk.owns_lock ())
    lk.lock ();
  return c->sticky;
}

/* after the upload stream has been waited for: the scan's two arrays apart */
static void
unpack_scan (Up &u)
{
  if (u.raw.empty ())
    return;
  const size_t h = (size_t) u.rr.h;
  u.spans.resize (h);
  u.groups.resize (h);
  memcpy (u.spans.data (), u.raw.data (), h * sizeof (int2));
  memcpy (u.groups.data (), u.raw.data () + 2 * h, h * sizeof (int));
  u.raw.clear ();
}

/* One uploaded rectangle becomes a box of the overlay: cropped to its non-transparent row runs
 * (or kept whole without auto-crop), with the sparsity figures of what remains. */
static void
append_box (Ctx *c, Overlay *ov, Up &u, size_t n_boxes)
{
  unpack_scan (u);
  OverlayBox box;
  box.declared = { u.rr.x, u.rr.y, u.rr.w, u.rr.h };
  box.first_rect = (uint32_t) ov->rects.size ();
  box.ga = u.rr.ga;
  box.slot = u.slot;
  box.src = u.src;
  if (!c->autocrop) {
    ov->rects.push_back (u.rr);
  } else {
    std::vector<FlucTtmlBlendRect> subs;
    /* at most 8 runs per rectangle, and never more sub-rectangles than the 64-bit band masks hold */
    crop_runs (u.spans, 16, std::max<size_t> (1, std::min<size_t> (8, FLUC_TTMLBLEND_MAX_RECTANGLES / std::max<size_t> (1, n_boxes))), subs);
    for (const FlucTtmlBlendRect &s : subs) {
      /* how sparse is what remains after the crop: 16-pixel groups with some alpha against
       * all groups of the kept sub-rectangles */
      box.groups_all += (uint64_t) ceil_div (s.w, 16) * (uint64_t) s.h;
      for (int y = s.y; y < s.y + s.h; y++) {
        box.groups_on += (uint64_t) (u.groups[y] & 0xffff);
        box.groups_opaque += (uint64_t) (u.groups[y] >> 16);
      }
      RawRect q = u.rr;
      q.dev = u.rr.dev + (size_t) s.y * u.rr.pitch + (size_t) s.x * 4;
      q.x = u.rr.x + s.x;
      q.y = u.rr.y + s.y;
      q.w = s.w;
      q.h = s.h;
      ov->rects.push_back (q);
    }
  }
  box.n_rects = (uint32_t) ov->rects.size () - box.first_rect;
  ov->boxes.push_back (box);
}

/* Text without a background box leaves most 16-byte vectors under the cue untouched, and
 * under an opaque box (alpha 255) the result does not depend on the frame at all. In place
 * (dst == src, host frames over PCIe) it then pays to look at the overlay before touching
 * the frame: transparent vectors are skipped, opaque ones are written without being read.
 * Under a translucent box it costs latency for nothing (tools/lazy_probe.py).
 * FLUC_TTMLBLEND_LAZY=0/1 forces it. */
static void
decide_lazy (Overlay *ov)
{
  static const char *lazy_env = getenv ("FLUC_TTMLBLEND_LAZY");
  uint64_t groups_all = 0, groups_on = 0, groups_opaque = 0;
  for (const OverlayBox &b : ov->boxes) {
    /* what the blend sees: a box at global alpha 0 is transparent, only one at 1 has opaque vectors */
    groups_all += b.groups_all;
    groups_on += b.ga ? b.groups_on : 0;
    groups_opaque += b.ga == 255 ? b.groups_opaque : 0;
  }
  ov->transparent_fraction = groups_all ? 1.0 - (double) groups_on / (double) groups_all : 0.0;
  ov->opaque_fraction = groups_all ? (double) groups_opaque / (double) groups_all : 0.0;
  ov->lazy_inplace = lazy_env ? atoi (lazy_env) != 0 : ov->transparent_fraction + ov->opaque_fraction >= 0.3;
  /* out of place every vector is written anyway; what can be saved is the read under an opaque
   * box (FLUC_TTMLBLEND_OPAQUE_SKIP=0/1 forces it) */
  static const char *skip_env = getenv ("FLUC_TTMLBLEND_OPAQUE_SKIP");
  ov->opaque_skip = skip_env ? atoi (skip_env) != 0 : ov->opaque_fraction >= 0.3;
}

/* Waits for uploads and scans, crops every rectangle to its non-transparent row runs and
 * swaps the stream's overlay. */
static int
finish_install (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, std::shared_ptr<Overlay> ov,
    std::vector<Up> &ups, const InstallStats &st)
{
  int rc = wait_uploads (c, lk);
  if (rc)
    return rc;
  c->stats.h2d_bytes += st.h2d_bytes;
  c->stats.prepare_launches += st.launches;
  for (Up &u : ups)
    append_box (c, ov.get (), u, ups.size ());
  if (ov->rects.size () > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  decide_lazy (ov.get ());
  /* The stream's frames will very likely keep the format and size they had: prepare the new
   * cue for them now, on the upload stream, so that the first frame after a cue change only
   * has an event to wait for instead of the prepare launches in front of it. */
  auto prev = c->overlays.find (stream);
  if (prev != c->overlays.end () && c->eager_prepare) {
    for (auto &p : prev->second->prepared) {
      if (!p->used || p->chroma_average != c->chroma_average)
        continue;
      Prepared *unused = nullptr;
      if ((rc = prepare_overlay (c, ov.get (), p->format, p->W, p->H, &unused)))
        return rc;
    }
  }
  c->overlays[stream] = ov;       /* frames already queued keep the old one */
  c->stats.overlays_set++;
  return 0;
}

/* gst_video_blend_scale_linear_RGBA's vertical pass, row by row: upstream keeps the
 * horizontally resampled source lines in a two-line cache (slot = row & 1) and tracks with
 * `y1` how far it has resampled. Simulating that bookkeeping here gives, for every
 * destination row, the two source rows and the 8-bit weight the kernel merges -- including
 * the rows where the cache holds something else than rows j and j+1 (docs/BLENDSPEC.md
 * section 10). */
std::vector<int4>
scale_row_plan (int src_h, int dst_h)
{
  const int y_inc = dst_h == 1 ? 0 : ((src_h - 1) << 16) / (dst_h - 1) - 1;
  int slot[2] = { 0, 0 };
  int y1 = 0, acc = 0;
  std::vector<int4> plan ((size_t) dst_h);
  for (int i = 0; i < dst_h; i++) {
    const int j = acc >> 16, x = acc & 0xffff;
    if (x == 0) {
      plan[i] = make_int4 (slot[j & 1], slot[j & 1], 0, 0);       /* memcpy of LINE (j) */
    } else {
      if (j > y1) {
        slot[j & 1] = j;
        y1++;
      }
      if (j >= y1) {
        slot[(j + 1) & 1] = j + 1;
        y1++;
      }
      plan[i] = make_int4 (slot[j & 1], slot[(j + 1) & 1], x >> 8, 0);
    }
    acc += y_inc;
  }
  return plan;
}

int
overlay_install (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, const FlucTtmlBlendRectangle *rects,
    uint32_t n, int image_w, int image_h)
{
  NvtxRange nvtx ("ttmlblend.overlay_set");
  for (uint32_t i = 0; i < n; i++) {
    const FlucTtmlBlendRectangle &r = rects[i];
    if (!r.pixels || r.width <= 0 || r.height <= 0 || r.stride < r.width * 4 || r.render_width < 0 ||
        r.render_height < 0 || r.render_width > 32768 || r.render_height > 32768)
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
    const int rw = r.render_width ? r.render_width : r.width, rh = r.render_height ? r.render_height : r.height;
    if ((rw != r.width || rh != r.height) && (r.width < 2 || r.height < 2))
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;   /* upstream reads outside the image here */
    /* the scaler's 16.16 positions ((side - 1) << 16, x * x_inc, the row plan's accumulator)
     * are 32-bit: past 32768 on a side they overflow (upstream's gint arithmetic is undefined
     * there too) and the kernel would read outside the source */
    if ((rw != r.width || rh != r.height) && (r.width > 32768 || r.height > 32768 || rw > 32768 || rh > 32768))
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  }
  std::shared_ptr<Overlay> ov (new Overlay ());
  ov->ctx = c;
  /* image_w > 0: the rectangles are the (disjoint) region boxes of one image of that size at
   * the frame's origin -- the ttmlrender form, which overlay_update can patch later */
  ov->image_w = image_w;
  ov->image_h = image_h;
  ov->updatable = image_w > 0 && image_h > 0;
  ov->movable = !ov->updatable;
  ov->n_alphas = std::max<uint32_t> (1, n);
  std::vector<Up> ups;
  std::vector<std::vector<int4>> plans;     /* host side of async uploads: alive until finish_install */
  InstallStats st;
  /* Uploading (a copy from pageable memory holds the caller for its whole length), scaling and
   * scanning touch only this overlay-to-be and the upload stream: the context is unlocked
   * meanwhile, so a cue change of one stream does not stall the frames of all the others. Any
   * failure takes the lock back before it reports (CUU). */
  lk.unlock ();
  for (uint32_t i = 0; i < n; i++) {
    const FlucTtmlBlendRectangle &r = rects[i];
    /* gst_video_overlay_rectangle_needs_scaling: render size != pixel size */
    const int rw = r.render_width ? r.render_width : r.width, rh = r.render_height ? r.render_height : r.height;
    const bool scaled = rw != r.width || rh != r.height;
    /* gst_video_blend: negative offsets skip source columns / rows. The composition form keeps
     * them on the device all the same, clipped at prepare time (rect_params), so that
     * overlay_set_positions can bring them into the frame later. */
    const int xoff = (!ov->movable && r.x < 0) ? -r.x : 0, yoff = (!ov->movable && r.y < 0) ? -r.y : 0;
    if (xoff >= rw || yoff >= rh)
      continue;
    Up u;
    u.slot = i;
    RawRect &rr = u.rr;
    rr.w = rw - xoff;
    rr.h = rh - yoff;
    rr.x = r.x + xoff;
    rr.y = r.y + yoff;
    rr.ga = (int) (255.0 * r.global_alpha);
    rr.ga = std::max (0, std::min (255, rr.ga));
    rr.premul = (r.flags & FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA) != 0;
    ov->declared.push_back ({ rr.x, rr.y, rr.w, rr.h });
    int rc;
    if (!scaled) {
      if ((rc = upload_rect (c, lk, r.pixels + (size_t) yoff * r.stride + (size_t) xoff * 4, r.stride, rr, st)))
        return rc;
      if (ov->movable)
        u.src = { rr.block, rr.dev, rr.pitch, rr.w, rr.h, rr.premul };
    } else {
      /* the whole source goes up, is scaled to the render size on the GPU, and the clipped
       * part of the scaled image is what gets blended */
      const int sp = (int) align_up ((size_t) r.width * 4, 256);
      void *s = nullptr, *d = nullptr, *p = nullptr;
      CUU (c, lk, cudaMallocFromPoolAsync (&s, (size_t) sp * r.height, c->mem_pool, c->up_stream));
      CUU (c, lk, cudaMemcpy2DAsync (s, sp, r.pixels, r.stride, (size_t) r.width * 4, r.height,
              cudaMemcpyDefault, c->up_stream));
      if (!on_device (r.pixels))
        st.h2d_bytes += (uint64_t) r.width * 4 * r.height;
      plans.push_back (scale_row_plan (r.height, rh));
      CUU (c, lk, cudaMallocFromPoolAsync (&p, (size_t) rh * sizeof (int4), c->mem_pool, c->up_stream));
      CUU (c, lk, cudaMemcpyAsync (p, plans.back ().data (), (size_t) rh * sizeof (int4), cudaMemcpyHostToDevice,
              c->up_stream));
      rr.pitch = (int) align_up ((size_t) rw * 4, 256);
      CUU (c, lk, cudaMallocFromPoolAsync (&d, (size_t) rr.pitch * rh, c->mem_pool, c->up_stream));
      rr.block = make_block (c, d);
      const int x_inc = rw == 1 ? 0 : ((r.width - 1) << 16) / (rw - 1) - 1;
      CUU (c, lk, launch_scale (static_cast<const uint8_t *> (s), sp, static_cast<const int4 *> (p), x_inc,
              static_cast<uint8_t *> (d), rr.pitch, rw, rh, c->up_stream));
      st.launches++;
      /* the composition form keeps the source for overlay_set_render_rectangles */
      if (ov->movable)
        u.src = { make_block (c, s), static_cast<const uint8_t *> (s), sp, r.width, r.height, rr.premul };
      else
        CUU (c, lk, cudaFreeAsync (s, c->up_stream));
      CUU (c, lk, cudaFreeAsync (p, c->up_stream));
      rr.dev = static_cast<uint8_t *> (d) + (size_t) yoff * rr.pitch + (size_t) xoff * 4;
    }
    if ((rc = scan_rows (c, lk, u)))
      return rc;
    ups.push_back (std::move (u));
  }
  return finish_install (c, lk, stream, ov, ups, st);
}

/* overlay_update: the stream's cue changed inside `changed` only (a <set> animation step, a
 * roll-up line: the producer re-renders its whole image for every timeline event,
 * /root/reference/plugins/ttml/gstttmlrender.c:1442-1452, /root/reference/plugins/ttml/gstttmlevent.c:208-233).
 * Boxes of the current overlay that the changed rectangles do not touch keep their device
 * pixels, their crop and their prepared planes -- the new overlay shares those blocks with the
 * old one -- and only the touched boxes are uploaded, scanned and prepared again. Returns
 * FLUC_TTMLBLEND_ERROR_NOT_FOUND when there is nothing to patch (no overlay from overlay_set of
 * the same image size, or a change outside every box): the caller installs the image whole. */
int
overlay_update_image (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, const uint8_t *bgra, int w, int h,
    int stride, const FlucTtmlBlendRect *changed, uint32_t n_changed)
{
  NvtxRange nvtx ("ttmlblend.overlay_update");
  auto it = c->overlays.find (stream);
  if (it == c->overlays.end () || !it->second->updatable || it->second->image_w != w || it->second->image_h != h)
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  std::shared_ptr<Overlay> old = it->second;
  std::vector<bool> touched (old->boxes.size (), false);
  size_t n_touched = 0;
  for (uint32_t k = 0; k < n_changed; k++) {
    const int x0 = std::max (changed[k].x, 0), y0 = std::max (changed[k].y, 0);
    const int x1 = std::min (changed[k].x + changed[k].w, w), y1 = std::min (changed[k].y + changed[k].h, h);
    if (x1 <= x0 || y1 <= y0)
      continue;
    /* the boxes are disjoint: the change lies inside them iff the intersections add up to it */
    uint64_t covered = 0;
    for (size_t b = 0; b < old->boxes.size (); b++) {
      const FlucTtmlBlendRect &d = old->boxes[b].declared;
      const int ix0 = std::max (x0, d.x), iy0 = std::max (y0, d.y);
      const int ix1 = std::min (x1, d.x + d.w), iy1 = std::min (y1, d.y + d.h);
      if (ix1 > ix0 && iy1 > iy0) {
        covered += (uint64_t) (ix1 - ix0) * (uint64_t) (iy1 - iy0);
        if (!touched[b]) {
          touched[b] = true;
          n_touched++;
        }
      }
    }
    if (covered != (uint64_t) (x1 - x0) * (uint64_t) (y1 - y0))
      return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  }
  if (n_touched == 0)
    return 0;                   /* nothing changed */

  /* upload + scan of the touched boxes, context unlocked (as in overlay_install) */
  std::vector<Up> ups (old->boxes.size ());
  InstallStats st;
  lk.unlock ();
  for (size_t b = 0; b < old->boxes.size (); b++) {
    if (!touched[b])
      continue;
    const FlucTtmlBlendRect &d = old->boxes[b].declared;
    RawRect &rr = ups[b].rr;
    rr.x = d.x; rr.y = d.y; rr.w = d.w; rr.h = d.h;
    rr.ga = 255;
    rr.premul = true;
    int rc;
    if ((rc = upload_rect (c, lk, bgra + (size_t) d.y * stride + (size_t) d.x * 4, stride, rr, st)) ||
        (rc = scan_rows (c, lk, ups[b])))
      return rc;
  }
  int rc = wait_uploads (c, lk);
  if (rc)
    return rc;
  auto now = c->overlays.find (stream);
  if (now == c->overlays.end () || now->second != old)
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;      /* replaced meanwhile by another thread */
  c->stats.h2d_bytes += st.h2d_bytes;

  std::shared_ptr<Overlay> nv (new Overlay ());
  nv->ctx = c;
  nv->image_w = w;
  nv->image_h = h;
  nv->updatable = true;
  nv->n_alphas = old->n_alphas;
  nv->declared = old->declared;
  std::vector<int> from_old;    /* new rectangle -> the old overlay's rectangle it is, or -1 */
  for (size_t b = 0; b < old->boxes.size (); b++) {
    if (touched[b]) {
      /* new pixels, prepared without a global alpha (but averaged chroma); the box keeps its
       * current one */
      ups[b].slot = old->boxes[b].slot;
      ups[b].rr.ga = old->boxes[b].ga;
      append_box (c, nv.get (), ups[b], old->boxes.size ());
      for (uint32_t k = nv->boxes.back ().first_rect; k < nv->rects.size (); k++)
        nv->rects[k].ga = 255;
      from_old.resize (nv->rects.size (), -1);
    } else {
      OverlayBox box = old->boxes[b];
      box.first_rect = (uint32_t) nv->rects.size ();
      for (uint32_t k = 0; k < old->boxes[b].n_rects; k++) {
        nv->rects.push_back (old->rects[old->boxes[b].first_rect + k]);
        from_old.push_back ((int) (old->boxes[b].first_rect + k));
      }
      nv->boxes.push_back (box);
    }
  }
  if (nv->rects.size () > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  decide_lazy (nv.get ());
  /* prepared for the formats / sizes the stream's frames have been using: kept rectangles bring
   * their prepared planes along, the others are prepared now */
  for (auto &p : old->prepared) {
    if (!p->used || p->chroma_average != c->chroma_average)
      continue;
    if ((rc = build_prepared (c, nv.get (), p->format, p->W, p->H, p->chroma_average, old.get (), p.get (),
             &from_old)))
      return rc;
  }
  c->overlays[stream] = nv;       /* frames already queued keep the old one */
  c->stats.overlays_set++;
  c->stats.overlays_updated++;
  return 0;
}

/* A new generation of ov: the same rectangles, boxes and form, nothing prepared yet. */
static std::shared_ptr<Overlay>
next_generation (const Overlay *ov)
{
  std::shared_ptr<Overlay> nv (new Overlay ());
  nv->ctx = ov->ctx;
  nv->rects = ov->rects;
  nv->boxes = ov->boxes;
  nv->declared = ov->declared;
  nv->image_w = ov->image_w;
  nv->image_h = ov->image_h;
  nv->updatable = ov->updatable;
  nv->movable = ov->movable;
  nv->n_alphas = ov->n_alphas;
  return nv;
}

/* Prepares nv, a new generation of the stream's overlay `old`, for everything old was prepared
 * for (build_prepared), and swaps it in. from_old maps nv's rectangles to old's (nullptr: the
 * same rectangles in the same order). */
static int
install_generation (Ctx *c, uint32_t stream, const Overlay *old, const std::shared_ptr<Overlay> &nv, bool batched,
    const std::vector<int> *from_old = nullptr)
{
  decide_lazy (nv.get ());
  std::vector<int> same;
  if (!from_old) {
    same.resize (nv->rects.size ());
    std::iota (same.begin (), same.end (), 0);
    from_old = &same;
  }
  for (auto &p : old->prepared) {
    const int rc = build_prepared (c, nv.get (), p->format, p->W, p->H, p->chroma_average, old, p.get (), from_old,
        batched);
    if (rc)
      return rc;
  }
  c->overlays[stream] = nv;       /* frames already queued keep the old one */
  return 0;
}

/* overlay_set_global_alpha: a new generation of the stream's overlay that differs from the
 * current one in its boxes' global alphas only. It shares every device block -- raw pixels and
 * prepared planes -- and brings new rectangle tables (a few hundred bytes, uploaded on the upload
 * stream and waited for through Prepared::ready like a cue change). Its layouts are built again
 * at the first frame and get the ids of equal band lists, so a fading stream's frames still share
 * launches. The PLANE8 kinds need the alpha bytes without a global alpha folded in: a box
 * installed below 1 is prepared once more from its raw pixels the first time it changes.
 * Averaged 4:2:0 chroma (chroma_average) holds the value itself: it is prepared again, alone,
 * for every box whose value changed. */
int
overlay_set_alpha (Ctx *c, uint32_t stream, const int *ga, uint32_t n)
{
  NvtxRange nvtx ("ttmlblend.overlay_set_global_alpha");
  auto it = c->overlays.find (stream);
  if (it == c->overlays.end ())
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  const std::shared_ptr<Overlay> old = it->second;
  if (n != 1 && n != old->n_alphas)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  std::shared_ptr<Overlay> nv = next_generation (old.get ());
  bool changed = false;
  for (OverlayBox &b : nv->boxes) {
    const int v = ga[n == 1 ? 0 : b.slot];
    if (v == b.ga)
      continue;
    changed = true;
    b.ga = v;
    for (uint32_t i = b.first_rect; i < b.first_rect + b.n_rects; i++)
      nv->rects[i].ga = 255;    /* from now on the blend applies it */
  }
  if (!changed)
    return 0;
  return install_generation (c, stream, old.get (), nv, false);
}

/* overlay_set_positions: a new generation of the stream's overlay whose boxes sit at (x[i], y[i])
 * (box i = rectangle i of overlay_set_rectangles). It shares every raw block; the crop runs are in
 * the rectangle's own coordinates and move with it. What depends on the position -- the shift
 * onto each destination plane's 16-byte grid, the chroma siting, the clipping at the frame
 * edges -- is prepared again from the resident pixels for every moved rectangle: one batch launch
 * per (format, size) the old generation was prepared for, on the upload stream, waited for through
 * Prepared::ready like a cue change. Global alphas carry over; averaged 4:2:0 chroma is prepared
 * again at the box's current value by its own kernel. Rectangles that stay keep their planes. */
int
overlay_set_positions (Ctx *c, uint32_t stream, const int32_t *x, const int32_t *y, uint32_t n)
{
  NvtxRange nvtx ("ttmlblend.overlay_set_positions");
  auto it = c->overlays.find (stream);
  if (it == c->overlays.end ())
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  const std::shared_ptr<Overlay> old = it->second;
  if (!old->movable || n != old->boxes.size ())
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  for (const OverlayBox &b : old->boxes)
    if ((int64_t) x[b.slot] + b.declared.w > INT32_MAX || (int64_t) y[b.slot] + b.declared.h > INT32_MAX)
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  std::shared_ptr<Overlay> nv = next_generation (old.get ());
  bool changed = false;
  for (OverlayBox &b : nv->boxes) {
    const int bx = x[b.slot], by = y[b.slot];
    if (bx == b.declared.x && by == b.declared.y)
      continue;
    changed = true;
    for (uint32_t i = b.first_rect; i < b.first_rect + b.n_rects; i++) {
      RawRect &rr = nv->rects[i];
      rr.x = bx + (rr.x - b.declared.x);      /* the crop run's offset inside the rectangle */
      rr.y = by + (rr.y - b.declared.y);
    }
    b.declared.x = bx;
    b.declared.y = by;
    nv->declared[b.slot] = b.declared;
  }
  if (!changed)
    return 0;
  return install_generation (c, stream, old.get (), nv, true);
}

/* overlay_set_render_rectangles: a new generation of the stream's overlay whose boxes sit at
 * render[i] and are render[i].w x render[i].h (box i = rectangle i of overlay_set_rectangles; a
 * side of 0: the pixel size). A box whose size stays is moved as overlay_set_positions moves it.
 * A resized box is built again from its resident source (BoxSource): scaled into a new block of
 * the render size, or the source itself at its pixel size, and cropped by a fresh row scan exactly
 * as overlay_install crops -- every resized box in one launch of the scale-and-scan kernel, one
 * upload of the row plans and one readback of the spans, waited for with the context unlocked.
 * Its new pixels are prepared like a box an update touches (the box keeps its global alpha, the
 * blend applies it), with the moved boxes in one batch launch per (format, size) the old generation
 * was prepared for. */
int
overlay_set_render (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, const FlucTtmlBlendRect *render,
    uint32_t n)
{
  NvtxRange nvtx ("ttmlblend.overlay_set_render_rectangles");
  auto it = c->overlays.find (stream);
  if (it == c->overlays.end ())
    return FLUC_TTMLBLEND_ERROR_NOT_FOUND;
  const std::shared_ptr<Overlay> old = it->second;
  if (!old->movable || n != old->boxes.size ())
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  /* the limits overlay_install applies to a scaled rectangle */
  for (const OverlayBox &b : old->boxes) {
    const FlucTtmlBlendRect &r = render[b.slot];
    if (r.w < 0 || r.h < 0 || r.w > 32768 || r.h > 32768)
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
    const int w = r.w ? r.w : b.src.w, h = r.h ? r.h : b.src.h;
    if ((w != b.src.w || h != b.src.h) && (b.src.w < 2 || b.src.h < 2 || b.src.w > 32768 || b.src.h > 32768))
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
    if ((int64_t) r.x + w > INT32_MAX || (int64_t) r.y + h > INT32_MAX)
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  }
  /* which boxes change size, which only move */
  std::vector<Up> ups (old->boxes.size ());
  std::vector<bool> resized (old->boxes.size (), false);
  bool changed = false;
  std::vector<ScaleScanItem> items;
  std::vector<size_t> item_box;             /* box of every item */
  std::vector<int4> plans;
  for (size_t k = 0; k < old->boxes.size (); k++) {
    const OverlayBox &b = old->boxes[k];
    const FlucTtmlBlendRect &r = render[b.slot];
    const int w = r.w ? r.w : b.src.w, h = r.h ? r.h : b.src.h;
    changed = changed || r.x != b.declared.x || r.y != b.declared.y;
    if (w == b.declared.w && h == b.declared.h)
      continue;
    changed = true;
    resized[k] = true;
    RawRect &rr = ups[k].rr;
    rr.x = r.x; rr.y = r.y; rr.w = w; rr.h = h;
    rr.premul = b.src.premul;
    ScaleScanItem si = {};
    si.w = w;
    si.h = h;
    if (w == b.src.w && h == b.src.h) {
      /* back at its pixel size: the source itself, scanned */
      rr.block = b.src.block;
      rr.dev = const_cast<uint8_t *> (b.src.dev);
      rr.pitch = b.src.pitch;
      si.src = b.src.dev;
      si.src_pitch = b.src.pitch;
      si.plan = -1;
      if (!c->autocrop)
        continue;
    } else {
      si.src = b.src.dev;
      si.src_pitch = b.src.pitch;
      si.plan = (int32_t) plans.size ();
      const std::vector<int4> p = scale_row_plan (b.src.h, h);
      plans.insert (plans.end (), p.begin (), p.end ());
      si.x_inc = w == 1 ? 0 : ((b.src.w - 1) << 16) / (w - 1) - 1;
      rr.pitch = (int) align_up ((size_t) w * 4, 256);
      si.dst_pitch = rr.pitch;
    }
    items.push_back (si);
    item_box.push_back (k);
  }
  if (!changed)
    return 0;                   /* nothing changed */

  if (!items.empty ()) {
    /* one allocation: the row plans and (beyond the inline limit) the items, uploaded in one
     * copy, then the spans and group counts of every row, read back in one copy */
    const uint32_t n_items = (uint32_t) items.size ();
    const uint32_t rows = scale_scan_batch_plan (items.data (), n_items);
    const size_t plan_bytes = plans.size () * sizeof (int4);
    const size_t item_bytes = n_items > kScaleScanBatchInline ? n_items * sizeof (ScaleScanItem) : 0;
    const size_t scan_bytes = c->autocrop ? (size_t) rows * (sizeof (int2) + sizeof (int)) : 0;
    std::vector<uint8_t> up (plan_bytes + item_bytes);
    std::vector<uint8_t> back (scan_bytes);
    lk.unlock ();               /* as in overlay_update_image: this call's blocks and the upload stream only */
    for (size_t i = 0; i < items.size (); i++) {
      if (items[i].plan < 0)
        continue;
      RawRect &rr = ups[item_box[i]].rr;
      void *d = nullptr;
      CUU (c, lk, cudaMallocFromPoolAsync (&d, (size_t) rr.pitch * rr.h, c->mem_pool, c->up_stream));
      rr.block = make_block (c, d);
      rr.dev = static_cast<uint8_t *> (d);
      items[i].dst = rr.dev;
    }
    memcpy (up.data (), plans.data (), plan_bytes);
    if (item_bytes)
      memcpy (up.data () + plan_bytes, items.data (), item_bytes);
    void *buf = nullptr;
    CUU (c, lk, cudaMallocFromPoolAsync (&buf, std::max<size_t> (up.size () + scan_bytes, 16), c->mem_pool,
            c->up_stream));
    uint8_t *d = static_cast<uint8_t *> (buf);
    if (!up.empty ())
      CUU (c, lk, cudaMemcpyAsync (d, up.data (), up.size (), cudaMemcpyHostToDevice, c->up_stream));
    int2 *d_spans = scan_bytes ? reinterpret_cast<int2 *> (d + up.size ()) : nullptr;
    int *d_groups = scan_bytes ? reinterpret_cast<int *> (d_spans + rows) : nullptr;
    CUU (c, lk, launch_scale_scan_batch (items.data (), n_items,
            reinterpret_cast<const ScaleScanItem *> (d + plan_bytes), reinterpret_cast<const int4 *> (d), d_spans,
            d_groups, rows, c->up_stream));
    if (scan_bytes)
      CUU (c, lk, cudaMemcpyAsync (back.data (), d_spans, scan_bytes, cudaMemcpyDeviceToHost, c->up_stream));
    CUU (c, lk, cudaFreeAsync (buf, c->up_stream));
    int rc = wait_uploads (c, lk);
    if (rc)
      return rc;
    c->stats.prepare_launches++;
    if (scan_bytes) {
      const int2 *spans = reinterpret_cast<const int2 *> (back.data ());
      const int *groups = reinterpret_cast<const int *> (spans + rows);
      for (size_t i = 0; i < items.size (); i++) {
        Up &u = ups[item_box[i]];
        u.spans.assign (spans + items[i].row0, spans + items[i].row0 + items[i].h);
        u.groups.assign (groups + items[i].row0, groups + items[i].row0 + items[i].h);
      }
    }
    auto now = c->overlays.find (stream);
    if (now == c->overlays.end () || now->second != old)
      return FLUC_TTMLBLEND_ERROR_NOT_FOUND;    /* replaced meanwhile by another thread */
  }

  std::shared_ptr<Overlay> nv = next_generation (old.get ());
  nv->rects.clear ();
  nv->boxes.clear ();
  std::vector<int> from_old;    /* new rectangle -> the old overlay's rectangle it is, or -1 */
  for (size_t k = 0; k < old->boxes.size (); k++) {
    const OverlayBox &b = old->boxes[k];
    if (resized[k]) {
      /* new pixels, prepared without a global alpha (but averaged chroma); the box keeps its current one */
      Up &u = ups[k];
      u.slot = b.slot;
      u.src = b.src;
      u.rr.ga = b.ga;
      append_box (c, nv.get (), u, old->boxes.size ());
      for (uint32_t i = nv->boxes.back ().first_rect; i < nv->rects.size (); i++)
        nv->rects[i].ga = 255;
      from_old.resize (nv->rects.size (), -1);
    } else {
      /* kept, or moved: the crop runs are offsets inside the rectangle (overlay_set_positions) */
      const FlucTtmlBlendRect &r = render[b.slot];
      OverlayBox box = b;
      box.first_rect = (uint32_t) nv->rects.size ();
      box.declared.x = r.x;
      box.declared.y = r.y;
      for (uint32_t i = b.first_rect; i < b.first_rect + b.n_rects; i++) {
        RawRect rr = old->rects[i];
        rr.x = r.x + (rr.x - b.declared.x);
        rr.y = r.y + (rr.y - b.declared.y);
        nv->rects.push_back (rr);
        from_old.push_back ((int) i);
      }
      nv->boxes.push_back (box);
    }
    nv->declared[b.slot] = nv->boxes.back ().declared;
  }
  if (nv->rects.size () > FLUC_TTMLBLEND_MAX_RECTANGLES)
    return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  return install_generation (c, stream, old.get (), nv, true, &from_old);
}

/* Cairo's colour conversion: double components -> premultiplied 16-bit shorts
 * (_cairo_color_compute_shorts: d * 65535.0 + 0.5) -> pixman a8r8g8b8 (short >> 8). */
static uint32_t
cairo_solid_pixel (uint32_t rgba8888)
{
  /* GET_CAIRO_COMP, /root/reference/plugins/ttml/gstttmlrender.c:1178 */
  const double r = ((rgba8888 >> 24) & 255) / 255.0, g = ((rgba8888 >> 16) & 255) / 255.0;
  const double b = ((rgba8888 >> 8) & 255) / 255.0, a = (rgba8888 & 255) / 255.0;
  const uint32_t as = (uint16_t) (a * 65535.0 + 0.5), rs = (uint16_t) (r * a * 65535.0 + 0.5);
  const uint32_t gs = (uint16_t) (g * a * 65535.0 + 0.5), bs = (uint16_t) (b * a * 65535.0 + 0.5);
  return ((as >> 8) << 24) | ((rs >> 8) << 16) | ((gs >> 8) << 8) | (bs >> 8);
}

/* The overlay composed on the GPU from region descriptors (SURVEY.md section 8f rank 3):
 * a cleared frame-sized canvas, every region drawn onto it in list order by
 * ttmlblend_region_kernel, then installed like an uploaded image cropped to the boxes. */
int
overlay_install_regions (Ctx *c, std::unique_lock<std::mutex> &lk, uint32_t stream, int W, int H,
    const FlucTtmlBlendRegion *regions, uint32_t n)
{
  NvtxRange nvtx ("ttmlblend.overlay_set_regions");
  for (uint32_t i = 0; i < n; i++)
    if (regions[i].w <= 0 || regions[i].h <= 0 || !(regions[i].opacity >= 0.0 && regions[i].opacity <= 1.0) ||
        (regions[i].layer && regions[i].layer_stride < 4 * regions[i].w))
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  {
    std::vector<FlucTtmlBlendRect> boxes;
    for (uint32_t i = 0; i < n; i++) {
      const FlucTtmlBlendRegion &r = regions[i];
      const int x0 = std::max (r.x, 0), y0 = std::max (r.y, 0);
      const int x1 = std::min (r.x + r.w, W), y1 = std::min (r.y + r.h, H);
      if (x1 > x0 && y1 > y0 && (r.background_color || r.layer))
        boxes.push_back ({ x0, y0, x1 - x0, y1 - y0 });
    }
    if (disjoint_cover (boxes).size () > FLUC_TTMLBLEND_MAX_RECTANGLES)
      return FLUC_TTMLBLEND_ERROR_TOO_MANY_RECTANGLES;
  }
  std::shared_ptr<Overlay> ov (new Overlay ());
  ov->ctx = c;
  InstallStats st;
  lk.unlock ();                 /* as in overlay_install: only this overlay and the upload stream from here */
  const int pitch = (int) align_up ((size_t) W * 4, 256);
  void *canvas = nullptr;
  CUU (c, lk, cudaMallocFromPoolAsync (&canvas, (size_t) pitch * H, c->mem_pool, c->up_stream));
  std::shared_ptr<DevBlock> canvas_block = make_block (c, canvas);
  CUU (c, lk, cudaMemsetAsync (canvas, 0, (size_t) pitch * H, c->up_stream));   /* CAIRO_OPERATOR_CLEAR */
  std::vector<void *> layers;
  std::vector<FlucTtmlBlendRect> boxes;
  for (uint32_t i = 0; i < n; i++) {
    const FlucTtmlBlendRegion &r = regions[i];
    const int x0 = std::max (r.x, 0), y0 = std::max (r.y, 0);
    const int x1 = std::min (r.x + r.w, W), y1 = std::min (r.y + r.h, H);
    if (x1 <= x0 || y1 <= y0)
      continue;
    RegionParams p = {};
    p.canvas = static_cast<uint8_t *> (canvas);
    p.canvas_pitch = pitch;
    p.x = x0; p.y = y0; p.w = x1 - x0; p.h = y1 - y0;
    p.lx = x0 - r.x; p.ly = y0 - r.y;
    p.bg = r.background_color ? cairo_solid_pixel (r.background_color) : 0u;
    p.m8 = r.opacity < 1.0 ? ((uint32_t) (uint16_t) (r.opacity * 65535.0 + 0.5)) >> 8 : 255u;
    if (r.layer) {
      const int lp = (int) align_up ((size_t) r.w * 4, 256);
      void *d = nullptr;
      CUU (c, lk, cudaMallocFromPoolAsync (&d, (size_t) lp * r.h, c->mem_pool, c->up_stream));
      layers.push_back (d);
      CUU (c, lk, cudaMemcpy2DAsync (d, lp, r.layer, r.layer_stride, (size_t) r.w * 4, r.h,
              cudaMemcpyDefault, c->up_stream));
      if (!on_device (r.layer))
        st.h2d_bytes += (uint64_t) r.w * 4 * r.h;
      p.layer = static_cast<uint8_t *> (d);
      p.layer_pitch = lp;
    }
    if (!p.bg && !p.layer)
      continue;                 /* nothing to draw */
    CUU (c, lk, launch_region (p, c->up_stream));
    st.launches++;
    boxes.push_back ({ x0, y0, x1 - x0, y1 - y0 });
  }
  for (void *d : layers)
    CUU (c, lk, cudaFreeAsync (d, c->up_stream));
  std::vector<Up> ups;
  for (const FlucTtmlBlendRect &b : disjoint_cover (boxes)) {
    Up u;
    u.rr.block = canvas_block;
    u.rr.dev = static_cast<uint8_t *> (canvas) + (size_t) b.y * pitch + (size_t) b.x * 4;
    u.rr.pitch = pitch;
    u.rr.w = b.w; u.rr.h = b.h; u.rr.x = b.x; u.rr.y = b.y;
    u.rr.ga = 255;
    u.rr.premul = true;
    ov->declared.push_back (b);
    int rc = scan_rows (c, lk, u);
    if (rc)
      return rc;
    ups.push_back (std::move (u));
  }
  return finish_install (c, lk, stream, ov, ups, st);
}

}  // namespace tbh
