/*
 * jobs.cu -- turns one frame into kernel work: planes are cut into bands at the rectangles'
 * edges and into windows left to right, each window gets its class (copy / one / bulk /
 * general); frames of equal geometry are collected into groups for the parameter-table kernel.
 */
#include "ttmlblend_internal.h"

namespace tbh {

int
check_frame (int fmt, int W, int H, const FlucTtmlBlendFrame *f)
{
  if (!f)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  if (!format_valid (fmt))
    return FLUC_TTMLBLEND_ERROR_UNSUPPORTED_FORMAT;
  if (W <= 0 || H <= 0 || W > 32768 || H > 32768)
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  for (int pl = 0; pl < format_planes (fmt); pl++)
    if (!f->plane[pl] || f->stride[pl] < plane_row_bytes (fmt, pl, W))
      return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  return 0;
}

void
push_window (std::vector<PlaneJob> &jobs, PlaneJob base, int v0, int v1, int y0, int y1)
{
  if (v1 <= v0 || y1 <= y0)
    return;
  const uint32_t nv = (uint32_t) (v1 - v0);
  /* magic division exactness: item * e < 2^32 with e = magic*nv - 2^32 < nv */
  const uint64_t magic = ((1ull << 32) + nv - 1) / nv;
  const uint64_t e = magic * nv - (1ull << 32);
  uint64_t max_items = e ? ((1ull << 32) - 1) / e : (1ull << 31);
  max_items = std::min<uint64_t> (max_items, 1ull << 31);
  int max_rows = (int) std::max<uint64_t> (1, std::min<uint64_t> (max_items / nv, 1 << 30));
  for (int r0 = y0; r0 < y1; r0 += max_rows) {
    PlaneJob j = base;
    j.win_v0 = v0;
    j.win_nv = (int32_t) nv;
    j.win_y0 = r0;
    j.win_rows = std::min (max_rows, y1 - r0);
    j.div_magic = (uint32_t) magic;     /* nv == 1 -> 2^32 truncates to 0; kernel special-cases it */
    const uint64_t items = (uint64_t) nv * (uint64_t) j.win_rows;
    j.n_chunks = (uint32_t) ((items + kItemsPerChunk - 1) / kItemsPerChunk);
    jobs.push_back (j);
  }
}

/* A window goes to the fast kernel where whole 16-byte vectors can be moved
 * (aligned frame, vector inside row_bytes); a ragged last vector column and
 * unaligned frames go to the byte-granular variant. */
void
push_split (std::vector<PlaneJob> &jobs, PlaneJob b, bool aligned, int v0, int v1, int y0, int y1)
{
  const int nv_full = b.row_bytes / 16;
  if (!aligned) {
    b.flags &= ~(JF_VECTOR | JF_FAST);
    push_window (jobs, b, v0, v1, y0, y1);
    return;
  }
  PlaneJob f = b;
  f.flags |= JF_VECTOR | JF_FAST;
  push_window (jobs, f, v0, std::min (v1, nv_full), y0, y1);
  if (v1 > nv_full) {
    PlaneJob t = b;
    t.flags = (t.flags | JF_VECTOR) & ~JF_FAST;
    push_window (jobs, t, std::max (v0, nv_full), v1, y0, y1);
  }
}

/* Builds the jobs of one frame: every plane is cut into bands of rows at the
 * top and bottom edges of the prepared rectangles, so that each band sees a
 * fixed set of rectangles and its class (copy / one rectangle / general) is
 * decided here, once, instead of per vector on the GPU. Returns the
 * algorithmic bytes moved (BASELINE.md section 2). */
uint64_t
build_jobs (int format, int W, int H, uint32_t frame_flags, const FlucTtmlBlendFrame *src,
    const FlucTtmlBlendFrame *dst, const Prepared *prep, bool windowed, std::vector<PlaneJob> &jobs)
{
  const int n_planes = format_planes (format);
  static const bool use_bulk = !getenv ("FLUC_TTMLBLEND_BULK") || atoi (getenv ("FLUC_TTMLBLEND_BULK")) != 0;
  /* windowed: only the vectors a rectangle covers are read and written (in
   * place, or host frames where untouched bytes never cross PCIe) */
  const bool inplace = windowed;
  uint64_t bytes = 0;
  std::vector<int> ys;
  for (int pl = 0; pl < n_planes; pl++) {
    PlaneJob b = {};
    b.src = static_cast<const uint8_t *> (src->plane[pl]);
    b.dst = static_cast<uint8_t *> (dst->plane[pl]);
    b.src_pitch = src->stride[pl];
    b.dst_pitch = dst->stride[pl];
    b.row_bytes = plane_row_bytes (format, pl, W);
    b.kind = plane_kind (format);
    b.plane = pl;
    const int rows = plane_rows (format, pl, H);
    const bool aligned = (((uintptr_t) b.src | (uintptr_t) b.dst | (uintptr_t) b.src_pitch |
            (uintptr_t) b.dst_pitch) & 15u) == 0;
    b.flags = (inplace ? JF_INPLACE : 0) |
        ((frame_flags & FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA) ? JF_DST_PREMUL : 0);
    static const std::vector<RectRef> none;
    const std::vector<RectRef> &rects = prep ? prep->h_rects[pl] : none;
    b.rects = prep ? prep->d_rects[pl] : nullptr;
    const int nv_row = ceil_div (b.row_bytes, 16);

    ys.clear ();
    ys.push_back (0);
    ys.push_back (rows);
    for (const RectRef &r : rects) {
      ys.push_back (std::max (0, std::min (rows, r.y0)));
      ys.push_back (std::max (0, std::min (rows, r.y1)));
    }
    std::sort (ys.begin (), ys.end ());
    ys.erase (std::unique (ys.begin (), ys.end ()), ys.end ());

    for (size_t bi = 0; bi + 1 < ys.size (); bi++) {
      const int ya = ys[bi], yb = ys[bi + 1];
      /* rectangles over this band, by first column; then cut the band into
       * windows left to right: gaps copy, a rectangle alone in its columns is
       * JC_ONE (no per-vector tests), rectangles sharing columns form one
       * JC_GENERAL window that applies them in blend order */
      struct InBand { int idx, v0, v1; };
      InBand in_band[FLUC_TTMLBLEND_MAX_RECTANGLES];
      int n_in = 0;
      for (size_t i = 0; i < rects.size (); i++) {
        const RectRef &r = rects[i];
        if (r.y0 <= ya && r.y1 >= yb && r.v0 < nv_row && r.v1 > 0)
          in_band[n_in++] = { (int) i, std::max (r.v0, 0), std::min (r.v1, nv_row) };
      }
      std::sort (in_band, in_band + n_in, [](const InBand &a, const InBand &c) { return a.v0 < c.v0; });
      auto emit = [&](int cls, unsigned long long mask, int one, int v0, int v1) {
        if (v1 <= v0)
          return;
        PlaneJob j = b;
        j.rect_mask = mask;
        j.one_rect = one < 0 ? 0 : one;
        j.cls = cls;
        /* prepared rows packed over exactly the window's columns: the overlay bytes of any
         * run of vectors of the band are contiguous -> TMA bulk staging in the group kernel */
        if (cls == JC_ONE && use_bulk && rects[one].v0 == v0 && rects[one].v1 == v1 &&
            rects[one].pitch == (v1 - v0) * 16 && (b.row_bytes & 15) == 0)
          j.cls = JC_ONE_BULK;
        push_split (jobs, j, aligned, v0, v1, ya, yb);
        bytes += 2ull * (uint64_t) std::min ((v1 - v0) * 16, b.row_bytes - v0 * 16) * (uint64_t) (yb - ya);
      };
      int cursor = 0;
      for (int i = 0; i < n_in;) {
        unsigned long long mask = 1ull << in_band[i].idx;
        int c0 = in_band[i].v0, c1 = in_band[i].v1, k = i + 1;
        while (k < n_in && in_band[k].v0 < c1) {      /* shares columns with the cluster */
          mask |= 1ull << in_band[k].idx;
          c1 = std::max (c1, in_band[k].v1);
          k++;
        }
        if (!inplace)
          emit (JC_COPY, 0, -1, cursor, c0);
        emit (k - i == 1 ? JC_ONE : JC_GENERAL, mask, in_band[i].idx, c0, c1);
        cursor = c1;
        i = k;
      }
      if (!inplace)
        emit (JC_COPY, 0, -1, cursor, nv_row);
    }
  }
  if (prep)
    bytes += 4ull * prep->overlay_px;
  return bytes;
}

/* Turns the fast jobs of a layout into a band list for the group kernels. */
void
make_groupable (Layout &L, bool lazy_inplace)
{
  size_t n_fast = 0;
  for (const PlaneJob &j : L.jobs)
    n_fast += (j.flags & JF_FAST) ? 1 : 0;
  if (n_fast == 0 || n_fast > (size_t) kMaxGroupBands)
    return;
  std::vector<PlaneJob> rest;
  uint32_t total = 0;
  int gflags = -1;
  for (const PlaneJob &j : L.jobs) {
    if (!(j.flags & JF_FAST)) {
      rest.push_back (j);
      continue;
    }
    BandDesc b = {};
    b.chunk_begin = total;
    b.plane = j.plane;
    b.win_v0 = j.win_v0;
    b.win_nv = j.win_nv;
    b.win_y0 = j.win_y0;
    b.win_rows = j.win_rows;
    b.div_magic = j.div_magic;
    b.cls = j.cls;
    b.one_rect = j.one_rect;
    b.rect_mask_lo = (uint32_t) j.rect_mask;
    b.rect_mask_hi = (uint32_t) (j.rect_mask >> 32);
    b.n_chunks = j.n_chunks;
    total += j.n_chunks;
    L.bands.push_back (b);
    gflags = j.flags & (JF_INPLACE | JF_DST_PREMUL);
  }
  /* frame = umulhi (chunk, ceil (2^32 / cpf)) must be exact for every chunk of a full group */
  const uint64_t magic = ((1ull << 32) + total - 1) / total;
  const uint64_t e = magic * total - (1ull << 32);
  if ((uint64_t) kMaxPlainGroupFrames * total * e >= (1ull << 32) ||
      (uint64_t) kMaxPlainGroupFrames * total >= (1ull << 26)) {
    L.bands.clear ();
    return;
  }
  /* `look`: the overlay is worth looking at before the frame is touched -- in place that skips
   * transparent vectors and does not read under opaque ones, out of place it does not read
   * under opaque ones (the caller picks the overlay's figure that goes with the frame) */
  if (lazy_inplace)
    gflags |= (gflags & JF_INPLACE) ? JF_LAZY : JF_OPAQUE;
  for (const PlaneJob &j : L.jobs)
    if (j.flags & JF_FAST)
      L.gjobs.push_back (j);
  L.jobs.swap (rest);
  L.grouped = true;
  L.chunks_per_frame = total;
  L.gflags = gflags;
}

static uint32_t
aligned_mask_of (int format, const FlucTtmlBlendFrame *src, const FlucTtmlBlendFrame *dst)
{
  uint32_t m = 0;
  for (int pl = 0; pl < format_planes (format); pl++)
    if ((((uintptr_t) src->plane[pl] | (uintptr_t) dst->plane[pl] | (uintptr_t) src->stride[pl] |
                (uintptr_t) dst->stride[pl]) & 15u) == 0)
      m |= 1u << pl;
  return m;
}

/* Layouts built for different overlays are different objects, but when every stream shows
 * the same kind of cue (same region box, filled background) their band lists are equal byte
 * for byte. Those get one id, found through a hash of the band list and confirmed by
 * comparing it, so that their frames share plain group launches. */
static uint64_t
canonical_layout_id (Ctx *c, const Layout &L)
{
  uint64_t h = 1469598103934665603ull;
  auto mix = [&h](const void *p, size_t n) {
    const uint8_t *b = static_cast<const uint8_t *> (p);
    for (size_t i = 0; i < n; i++)
      h = (h ^ b[i]) * 1099511628211ull;
  };
  mix (L.bands.data (), L.bands.size () * sizeof (BandDesc));
  mix (L.src_pitch, sizeof L.src_pitch);
  mix (L.dst_pitch, sizeof L.dst_pitch);
  mix (L.rect_off, sizeof L.rect_off);
  mix (&L.gflags, sizeof L.gflags);
  mix (&L.kind, sizeof L.kind);
  std::vector<Ctx::LayoutSig> &bucket = c->layout_sigs[h];
  for (const Ctx::LayoutSig &s : bucket)
    if (s.kind == L.kind && s.gflags == L.gflags && s.bands.size () == L.bands.size () &&
        memcmp (s.pitch, L.src_pitch, sizeof L.src_pitch) == 0 &&
        memcmp (s.pitch + 3, L.dst_pitch, sizeof L.dst_pitch) == 0 &&
        memcmp (s.rect_off, L.rect_off, sizeof L.rect_off) == 0 &&
        memcmp (s.bands.data (), L.bands.data (), L.bands.size () * sizeof (BandDesc)) == 0)
      return s.id;
  if (c->n_layout_sigs >= 4096) {       /* ids stay unique; equal layouts built later just get a new one */
    c->layout_sigs.clear ();
    c->n_layout_sigs = 0;
  }
  Ctx::LayoutSig s;
  s.id = L.id;
  s.kind = L.kind;
  s.gflags = L.gflags;
  memcpy (s.pitch, L.src_pitch, sizeof L.src_pitch);
  memcpy (s.pitch + 3, L.dst_pitch, sizeof L.dst_pitch);
  memcpy (s.rect_off, L.rect_off, sizeof L.rect_off);
  s.bands = L.bands;
  c->layout_sigs[h].push_back (std::move (s));
  c->n_layout_sigs++;
  return L.id;
}

/* The layout for this frame: found among those already built for the prepared overlay (or,
 * without an overlay, for the format and size), else built now. */
const Layout *
find_layout (Ctx *c, Prepared *prep, bool lazy_inplace, int format, int W, int H, uint32_t frame_flags,
    const FlucTtmlBlendFrame *src, const FlucTtmlBlendFrame *dst, bool windowed)
{
  std::vector<std::unique_ptr<Layout>> *list = nullptr;
  if (prep) {
    list = &prep->layouts;
  } else {
    for (auto &b : c->bare_layouts)
      if (b.format == format && b.W == W && b.H == H)
        list = &b.layouts;
    if (!list) {
      if (c->bare_layouts.size () >= 16) {
        launch_pending (c);               /* queued frames may point into what is dropped */
        c->bare_layouts.erase (c->bare_layouts.begin ());
      }
      c->bare_layouts.push_back ({ format, W, H, {} });
      list = &c->bare_layouts.back ().layouts;
    }
  }
  const uint32_t am = aligned_mask_of (format, src, dst);
  const uint32_t ff = frame_flags & FLUC_TTMLBLEND_FLAG_PREMULTIPLIED_ALPHA;
  const int n_planes = format_planes (format);
  for (auto &l : *list) {
    if (l->aligned_mask != am || l->windowed != windowed || l->frame_flags != ff)
      continue;
    bool same = true;
    for (int pl = 0; pl < n_planes; pl++)
      same = same && l->src_pitch[pl] == src->stride[pl] && l->dst_pitch[pl] == dst->stride[pl];
    if (same)
      return l.get ();
  }
  if (list->size () >= 8) {
    launch_pending (c);                   /* queued frames may point into what is dropped */
    list->erase (list->begin ());
  }
  std::unique_ptr<Layout> L (new Layout ());
  L->id = ++c->next_layout_id;
  L->kind = plane_kind (format);
  for (int pl = 0; pl < n_planes; pl++) {
    L->src_pitch[pl] = src->stride[pl];
    L->dst_pitch[pl] = dst->stride[pl];
  }
  L->aligned_mask = am;
  L->windowed = windowed;
  L->frame_flags = ff;
  L->algo_bytes = build_jobs (format, W, H, frame_flags, src, dst, prep, windowed, L->jobs);
  for (const PlaneJob &j : L->jobs)
    L->window_bytes += (uint64_t) std::min (j.win_nv * 16, j.row_bytes - j.win_v0 * 16) * (uint64_t) j.win_rows;
  for (int pl = 0; pl < 3; pl++)
    L->rect_off[pl] = prep ? prep->rect_off[pl] : 0;
  L->rects_all = prep ? prep->d_rects_all : nullptr;
  if (c->use_groups)
    make_groupable (*L, lazy_inplace);
  if (L->grouped)
    L->id = canonical_layout_id (c, *L);
  list->push_back (std::move (L));
  return list->back ().get ();
}

/* the rows a layout's windows touch, neighbouring bands of equal width merged */
void
layout_spans (const Layout *L, std::vector<StageSpan> &out)
{
  auto add = [&out](const PlaneJob &j) {
    StageSpan s;
    s.plane = j.plane;
    s.b0 = j.win_v0 * 16;
    s.nb = std::min (j.win_nv * 16, j.row_bytes - s.b0);
    s.y0 = j.win_y0;
    s.rows = j.win_rows;
    if (s.nb <= 0 || s.rows <= 0)
      return;
    for (StageSpan &o : out)
      if (o.plane == s.plane && o.b0 == s.b0 && o.nb == s.nb && o.y0 + o.rows == s.y0) {
        o.rows += s.rows;
        return;
      }
    out.push_back (s);
  };
  for (const PlaneJob &j : L->jobs)
    add (j);
  for (const PlaneJob &j : L->gjobs)
    add (j);
}

static FramePtrs
frame_ptrs (const PendingFrame &f)
{
  FramePtrs p = {};
  for (int pl = 0; pl < 3; pl++) {
    p.src[pl] = f.src[pl];
    p.dst[pl] = f.dst[pl];
  }
  p.rects = f.layout->rects_all;
  return p;
}

/* JF_GA for the frames whose prepared overlay leaves a global alpha to the blend: a launch that
 * holds one of them takes the kernel variant that scales the alpha bytes */
static int
frame_ga_flag (const PendingFrame &f)
{
  return f.prep && f.prep->fade ? JF_GA : 0;
}

/* The layout's table jobs with this frame's pointers, appended per (kind, fast). */
void
emit_table_jobs (const std::vector<PlaneJob> &tmpl, const PendingFrame &f, std::vector<PlaneJob> *by_kind)
{
  const int ga = frame_ga_flag (f);
  for (const PlaneJob &t : tmpl) {
    std::vector<PlaneJob> &v = by_kind[f.layout->kind * 2 + ((t.flags & JF_FAST) ? 1 : 0)];
    v.push_back (t);
    v.back ().src = f.src[t.plane];
    v.back ().dst = f.dst[t.plane];
    v.back ().flags |= ga;
  }
}

bool
group_accepts (const Group &g, const PendingFrame &f)
{
  return g.layout_id == f.layout->id && g.P.h.n_frames < (uint32_t) kMaxPlainGroupFrames;
}

void
group_start (Group &g, const PendingFrame &f)
{
  const Layout &L = *f.layout;
  memset (&g.P.h, 0, sizeof g.P.h);
  g.kind = L.kind;
  g.layout_id = L.id;
  g.dissolved = false;
  g.P.h.n_bands = (uint32_t) L.bands.size ();
  g.P.h.chunks_per_frame = L.chunks_per_frame;
  g.P.h.cpf_magic = (uint32_t) (((1ull << 32) + L.chunks_per_frame - 1) / L.chunks_per_frame);
  g.P.h.flags = L.gflags;
  memcpy (g.P.h.src_pitch, L.src_pitch, sizeof g.P.h.src_pitch);
  memcpy (g.P.h.dst_pitch, L.dst_pitch, sizeof g.P.h.dst_pitch);
  memcpy (g.P.h.rect_off, L.rect_off, sizeof g.P.h.rect_off);
  memcpy (g.P.bands, L.bands.data (), L.bands.size () * sizeof (BandDesc));
}

void
group_add (Group &g, const PendingFrame &f)
{
  g.P.frames[g.P.h.n_frames++] = frame_ptrs (f);
  g.P.h.flags |= frame_ga_flag (f);
}

void
multi_start (MultiGroup &m, const PendingFrame &f)
{
  const Layout &L = *f.layout;
  m.kind = L.kind;
  m.n_bands = 0;
  m.layouts.clear ();
  /* only the header: frames and bands are written as they are added */
  m.P.n_frames = 0;
  m.P.flags = L.gflags;
  memcpy (m.P.src_pitch, L.src_pitch, sizeof m.P.src_pitch);
  memcpy (m.P.dst_pitch, L.dst_pitch, sizeof m.P.dst_pitch);
  m.P.frame_begin[0] = 0;
}

/* Adds a groupable frame to a multi-layout launch if it fits: same kind, pitches and flags,
 * room for the frame and -- unless its band list is already there -- for its bands. */
bool
multi_add (MultiGroup &m, const PendingFrame &f)
{
  const Layout &L = *f.layout;
  MultiParams &P = m.P;
  if (m.kind != L.kind || (P.flags & ~JF_GA) != L.gflags || P.n_frames >= (uint32_t) kMaxGroupFrames ||
      memcmp (P.src_pitch, L.src_pitch, sizeof P.src_pitch) || memcmp (P.dst_pitch, L.dst_pitch, sizeof P.dst_pitch))
    return false;
  if ((uint64_t) P.frame_begin[P.n_frames] + L.chunks_per_frame >= (1ull << 26))
    return false;
  for (int pl = 0; pl < 3; pl++)
    if (L.rect_off[pl] < 0 || L.rect_off[pl] > 0xffff)
      return false;
  const size_t nb = L.bands.size ();
  int slot = -1;
  for (size_t i = 0; i < m.layouts.size (); i++)
    if (m.layouts[i].id == L.id) {
      slot = (int) i;
      break;
    }
  if (slot < 0) {
    if (m.n_bands + nb > (size_t) kMaxMultiBands)
      return false;
    memcpy (&P.bands[m.n_bands], L.bands.data (), nb * sizeof (BandDesc));
    m.layouts.push_back ({ L.id, (uint16_t) m.n_bands, (uint16_t) nb });
    slot = (int) m.layouts.size () - 1;
    m.n_bands += (uint32_t) nb;
  }
  const uint32_t k = P.n_frames++;
  P.frame_band0[k] = m.layouts[slot].band0;
  P.frame_nbands[k] = m.layouts[slot].n_bands;
  P.frames[k] = frame_ptrs (f);
  P.frames[k].pad_ = (uint64_t) L.rect_off[0] | ((uint64_t) L.rect_off[1] << 16) | ((uint64_t) L.rect_off[2] << 32);
  P.frame_begin[k + 1] = P.frame_begin[k] + L.chunks_per_frame;
  P.flags |= frame_ga_flag (f);
  return true;
}

}  // namespace tbh
