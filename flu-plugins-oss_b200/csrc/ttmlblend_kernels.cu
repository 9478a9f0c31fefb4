/*
 * ttmlblend_kernels.cu -- hand-written sm_100a kernels of the TTML overlay
 * blend: the per-frame blend and the once-per-cue overlay prepare.
 *
 * Arithmetic contract: docs/BLENDSPEC.md (gst-plugins-base video-blend.c /
 * video-format.c as named by BASELINE.json's north_star; SURVEY.md App. A).
 * Every formula below is the integer formula of that spec; nothing is
 * approximated. The kernels are HBM-bound byte work: 128-bit coalesced
 * loads/stores of the frame rows, overlay slices from the prepared cache
 * (L2-resident across the frames of a batch) staged through shared memory by
 * the TMA (cp.async.bulk + mbarrier), tables in kernel parameters, IDP.4A and
 * two-lane SIMD arithmetic for the blend itself, no tensor cores.
 *
 *   ttmlblend_group_kernel      frames of equal geometry, band list in parameters
 *   ttmlblend_blend_kernel      everything else (table in global memory, byte path)
 *   ttmlblend_prepare_kernel    once per cue: unpack, un-premultiply, BT.709, siting
 *   ttmlblend_prepare_chroma_avg_kernel   opt-in, non-parity 2x2 chroma mean
 *   ttmlblend_rowspan_kernel    once per cue: non-transparent span of every row
 *   ttmlblend_scale_scan_batch_kernel  once per resize: scale + row spans of every resized rectangle
 *   ttmlblend_blur_kernel       textOutline blur (pixman convolution semantics)
 */
#include "ttmlblend_kernels.cuh"

#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <utility>

namespace tb {

/* ---------------------------------------------------------------------- */
/* memory helpers                                                         */

__device__ __forceinline__ uint4
ld_frame16 (const uint8_t *p)
{
  uint4 r;
  asm volatile ("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
      : "=r" (r.x), "=r" (r.y), "=r" (r.z), "=r" (r.w) : "l" (p));
  return r;
}

__device__ __forceinline__ void
st_frame16 (uint8_t *p, const uint4 &v)
{
  asm volatile ("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};"
      :: "l" (p), "r" (v.x), "r" (v.y), "r" (v.z), "r" (v.w) : "memory");
}

/* prepared overlay: read-only for the kernel, re-read by every frame of the
 * batch, so keep it cacheable */
__device__ __forceinline__ uint4
ld_overlay16 (const uint8_t *p)
{
  return __ldg (reinterpret_cast<const uint4 *> (p));
}

template <typename T>
__device__ __forceinline__ T *
ldg_ptr (T *const *pp)
{
  return reinterpret_cast<T *> (__ldg (reinterpret_cast<const unsigned long long *> (pp)));
}

/* Fall-back for frames that are not 16-byte aligned and for the ragged tail of a row. GStreamer
 * only guarantees strides that are multiples of 4 (a 1366 or 854 pixel wide frame has 1368 /
 * 856 byte rows), so the 16 bytes of an item are moved with the widest accesses their address
 * allows -- two 64-bit, four 32-bit -- and byte by byte only where even that fails or the
 * row ends inside the item. */
__device__ __forceinline__ uint4
ld_frame_bytes (const uint8_t *p, int nvalid)
{
  uint32_t w[4] = { 0u, 0u, 0u, 0u };
  const uintptr_t a = reinterpret_cast<uintptr_t> (p);
  if (nvalid == 16 && (a & 7u) == 0) {
    const uint2 lo = *reinterpret_cast<const uint2 *> (p), hi = *reinterpret_cast<const uint2 *> (p + 8);
    return make_uint4 (lo.x, lo.y, hi.x, hi.y);
  }
  if ((a & 3u) == 0) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (4 * i + 4 <= nvalid) {
        w[i] = *reinterpret_cast<const uint32_t *> (p + 4 * i);
      } else {
#pragma unroll
        for (int b = 0; b < 4; b++)
          if (4 * i + b < nvalid)
            w[i] |= (uint32_t) p[4 * i + b] << (8 * b);
      }
    }
    return make_uint4 (w[0], w[1], w[2], w[3]);
  }
#pragma unroll
  for (int i = 0; i < 16; i++)
    if (i < nvalid)
      w[i >> 2] |= (uint32_t) p[i] << (8 * (i & 3));
  return make_uint4 (w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ void
st_frame_bytes (uint8_t *p, const uint4 &v, int nvalid)
{
  const uint32_t w[4] = { v.x, v.y, v.z, v.w };
  const uintptr_t a = reinterpret_cast<uintptr_t> (p);
  if (nvalid == 16 && (a & 7u) == 0) {
    *reinterpret_cast<uint2 *> (p) = make_uint2 (v.x, v.y);
    *reinterpret_cast<uint2 *> (p + 8) = make_uint2 (v.z, v.w);
    return;
  }
  if ((a & 3u) == 0) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (4 * i + 4 <= nvalid) {
        *reinterpret_cast<uint32_t *> (p + 4 * i) = w[i];
      } else {
#pragma unroll
        for (int b = 0; b < 4; b++)
          if (4 * i + b < nvalid)
            p[4 * i + b] = (uint8_t) (w[i] >> (8 * b));
      }
    }
    return;
  }
#pragma unroll
  for (int i = 0; i < 16; i++)
    if (i < nvalid)
      p[i] = (uint8_t) (w[i >> 2] >> (8 * (i & 3)));
}

/* ---------------------------------------------------------------------- */
/* programmatic dependent launch (JF_PDL / JF_DEP, ttmlblend_kernels.cuh) */

__device__ __forceinline__ void
pdl_begin (int flags)
{
  if (flags & JF_DEP)
    asm volatile ("griddepcontrol.wait;" ::: "memory");
  if (flags & JF_PDL)
    asm volatile ("griddepcontrol.launch_dependents;" ::: "memory");
}

/* a CTA's last act: grids complete in launch order, so "the previous grid has completed"
 * always means "everything launched before has completed" */
__device__ __forceinline__ void
pdl_end (int flags)
{
  if (flags & JF_PDL)
    asm volatile ("griddepcontrol.wait;" ::: "memory");
}

/* Launches `kernel` with or without the programmatic-serialisation attribute. */
template <typename... KArgs, typename... Args>
static cudaError_t
launch_ex (void (*kernel) (KArgs...), uint32_t grid, size_t smem, cudaStream_t stream, bool pdl, Args &&... args)
{
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3 (grid);
  cfg.blockDim = dim3 (kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx (&cfg, kernel, std::forward<Args> (args)...);
}

/* ---------------------------------------------------------------------- */
/* arithmetic                                                             */

/* PLANE8: four destination bytes. Opaque destination, straight source:
 *   out = (Cs * asrc + Cd * (255 - asrc)) / 255        (OVER00, adst = 255)
 * asrc == 0 leaves Cd untouched by the same formula, like the `continue`.
 * ~5.5 integer instructions per byte: the two products of a byte are one
 * IDP.4A ((Cs, Cd, 0, 0) . (a, 255 - a, ., .)), and the truncating /255 runs
 * on two 16-bit lanes at once, x / 255 == (x + 1 + (x >> 8)) >> 8 for
 * x <= 65534 (numerators are <= 255 * 255). */
__device__ __forceinline__ uint32_t
blend4_plane8 (uint32_t f, uint32_t a, uint32_t c)
{
  const uint32_t na = ~a;                               /* 255 - a, bytewise */
  const uint32_t cf01 = __byte_perm (c, f, 0x5140);     /* c0 f0 c1 f1 */
  const uint32_t cf23 = __byte_perm (c, f, 0x7362);     /* c2 f2 c3 f3 */
  const uint32_t an01 = __byte_perm (a, na, 0x5140);    /* a0 n0 a1 n1 */
  const uint32_t an23 = __byte_perm (a, na, 0x7362);    /* a2 n2 a3 n3 */
  const uint32_t n0 = __dp4a (cf01 & 0x0000ffffu, an01, 0u);
  const uint32_t n1 = __dp4a (cf01 & 0xffff0000u, an01, 0u);
  const uint32_t n2 = __dp4a (cf23 & 0x0000ffffu, an23, 0u);
  const uint32_t n3 = __dp4a (cf23 & 0xffff0000u, an23, 0u);
  uint32_t e = __byte_perm (n0, n2, 0x5410);            /* n0 | n2 << 16 */
  uint32_t o = __byte_perm (n1, n3, 0x5410);            /* n1 | n3 << 16 */
  e = e + ((e >> 8) & 0x00ff00ffu) + 0x00010001u;       /* quotients in bits 8-15, 24-31 */
  o = o + ((o >> 8) & 0x00ff00ffu) + 0x00010001u;
  return __byte_perm (e, o, 0x7351);                    /* q0 q1 q2 q3 */
}

__device__ __forceinline__ uint4
blend16_plane8 (uint4 f, const uint4 &a, const uint4 &c)
{
  if (a.x) f.x = blend4_plane8 (f.x, a.x, c.x);
  if (a.y) f.y = blend4_plane8 (f.y, a.y, c.y);
  if (a.z) f.z = blend4_plane8 (f.z, a.z, c.z);
  if (a.w) f.w = blend4_plane8 (f.w, a.w, c.w);
  return f;
}

/* PLANE8_RGB (24-bit RGB / BGR frames: no alpha byte, so adst = 255 and final_alpha = 255):
 * the same per-byte alpha / colour planes as PLANE8, but an RGB destination keeps the source's
 * premultiplied flag (BLENDSPEC section 2), so there are two operators per rectangle:
 *   straight source:       (Cs * asrc + Cd * (255 - asrc)) / 255           = the PLANE8 formula
 *   premultiplied source:  MIN (255, (Cs * ga + Cd * (255 - asrc)) / 255)
 * With ga == 255 the latter is Cs + (Cd * (255 - asrc)) / 255, saturating: the PLANE8 formula
 * on colour 0 plus a saturating byte add. ga < 255 needs 17-bit numerators: one byte at a time. */
__device__ __forceinline__ uint32_t
blend4_rgb24 (uint32_t f, uint32_t a, uint32_t c, uint32_t ga, bool sp)
{
  if (!sp)
    return blend4_plane8 (f, a, c);
  if (ga == 255u)
    return __vaddus4 (blend4_plane8 (f, a, 0u), c);      /* a == 0 bytes: f + 0 (their colour is 0) */
  uint32_t out = 0u;
#pragma unroll
  for (int k = 0; k < 32; k += 8) {
    const uint32_t as = (a >> k) & 0xffu, cs = (c >> k) & 0xffu, cd = (f >> k) & 0xffu;
    const uint32_t v = as ? min ((cs * ga + cd * (255u - as)) / 255u, 255u) : cd;
    out |= v << k;
  }
  return out;
}

__device__ __forceinline__ uint4
blend16_rgb24 (uint4 f, const uint4 &a, const uint4 &c, uint32_t ga, bool sp)
{
  if (a.x) f.x = blend4_rgb24 (f.x, a.x, c.x, ga, sp);
  if (a.y) f.y = blend4_rgb24 (f.y, a.y, c.y, ga, sp);
  if (a.z) f.z = blend4_rgb24 (f.z, a.z, c.z, ga, sp);
  if (a.w) f.w = blend4_rgb24 (f.w, a.w, c.w, ga, sp);
  return f;
}

/* The JF_GA variant of the PLANE8 kinds: the prepared alpha bytes hold the overlay's own alpha
 * and the rectangle's current global alpha is applied per frame, asrc = a * ga / 255 on every
 * byte (BLENDSPEC section 2), two 16-bit lanes per register as above (a * ga <= 65025). */
__device__ __forceinline__ uint32_t
scale4_alpha (uint32_t a, uint32_t ga)
{
  uint32_t e = (a & 0x00ff00ffu) * ga, o = ((a >> 8) & 0x00ff00ffu) * ga;
  e = e + ((e >> 8) & 0x00ff00ffu) + 0x00010001u;
  o = o + ((o >> 8) & 0x00ff00ffu) + 0x00010001u;
  return ((e >> 8) & 0x00ff00ffu) | (o & 0xff00ff00u);
}

__device__ __forceinline__ uint4
scale16_alpha (const uint4 &a, uint32_t ga)
{
  return make_uint4 (scale4_alpha (a.x, ga), scale4_alpha (a.y, ga), scale4_alpha (a.z, ga), scale4_alpha (a.w, ga));
}

/* kinds whose prepared overlay is an alpha byte plane + a colour byte plane */
__host__ __device__ constexpr bool
kind_is_planes (int kind)
{
  return kind == PK_PLANE8 || kind == PK_PLANE8_RGB;
}

/* PACKED: one pixel word, alpha in byte AP, the other three bytes colours.
 * gst_video_blend's BLENDLOOP with the four OVERxy operators. */
template <int AP>
__device__ __forceinline__ uint32_t
blend_px_packed (uint32_t f, uint32_t o, uint32_t ga, bool sp, bool dp)
{
  const uint32_t a = (o >> (8 * AP)) & 0xffu;
  const uint32_t asrc = (ga == 255u) ? a : (a * ga) / 255u;
  if (asrc == 0u)
    return f;
  const uint32_t adst = (f >> (8 * AP)) & 0xffu;
  const uint32_t na = 255u - asrc;
  uint32_t out;
  if (ga == 255u && adst == 255u && !dp) {
    /* opaque straight destination: final_alpha = 255. All four bytes at once on two 16-bit
     * lanes per register (even bytes / odd bytes); every lane stays <= 255 * 255, and
     * x / 255 == (x + 1 + (x >> 8)) >> 8 for x <= 65534. */
    const uint32_t fe = f & 0x00ff00ffu, fo = (f >> 8) & 0x00ff00ffu;
    uint32_t te, to;
    if (sp) {
      te = fe * na;                                   /* Cd * (255 - a) */
      to = fo * na;
    } else {
      te = (o & 0x00ff00ffu) * asrc + fe * na;        /* Cs * a + Cd * (255 - a) */
      to = ((o >> 8) & 0x00ff00ffu) * asrc + fo * na;
    }
    te = te + ((te >> 8) & 0x00ff00ffu) + 0x00010001u;
    to = to + ((to >> 8) & 0x00ff00ffu) + 0x00010001u;
    out = ((te >> 8) & 0x00ff00ffu) | (to & 0xff00ff00u);
    if (sp)
      /* OVER10: (Cs*255 + Cd*na)/255 = Cs + (Cd*na)/255, then MIN 255 -- a saturating byte
       * add; the alpha byte comes out as a + (255*na)/255 = 255 by itself */
      out = __vaddus4 (out, o);
    else
      out |= 0xffu << (8 * AP);
  } else {
    uint32_t fa = asrc + adst * na / 255u;
    out = fa << (8 * AP);
    if (fa == 0u)
      fa = 1u;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (k == AP)
        continue;
      const uint32_t cs = (o >> (8 * k)) & 0xffu;
      const uint32_t cd = (f >> (8 * k)) & 0xffu;
      uint32_t v;
      if (!dp)
        v = ((sp ? cs * ga : cs * asrc) + cd * adst * na / 255u) / fa;
      else
        v = ((sp ? cs * ga : cs * asrc) + cd * na) / 255u;
      out |= min (v, 255u) << (8 * k);
    }
  }
  return out;
}

/* One pixel of the common case -- global alpha 1, straight destination whose alpha byte is 255 --
 * without a branch: final_alpha = 255, and asrc == 0 falls out of the arithmetic (the weights
 * are 0 and 255, x * 255 / 255 is exact; a premultiplied source word with alpha 0 is all zero,
 * the prepare kernel sees to that). All four bytes at once on two 16-bit lanes per register
 * (even bytes / odd bytes); every lane stays <= 255 * 255, and
 * x / 255 == (x + 1 + (x >> 8)) >> 8 for x <= 65534. */
template <int AP>
__device__ __forceinline__ uint32_t
blend_px_packed_opaque (uint32_t f, uint32_t o, bool sp)
{
  const uint32_t a = (o >> (8 * AP)) & 0xffu, na = 255u - a;
  const uint32_t fe = f & 0x00ff00ffu, fo = (f >> 8) & 0x00ff00ffu;
  uint32_t te, to;
  if (sp) {
    te = fe * na;                                     /* Cd * (255 - a) */
    to = fo * na;
  } else {
    te = (o & 0x00ff00ffu) * a + fe * na;             /* Cs * a + Cd * (255 - a) */
    to = ((o >> 8) & 0x00ff00ffu) * a + fo * na;
  }
  te = te + ((te >> 8) & 0x00ff00ffu) + 0x00010001u;
  to = to + ((to >> 8) & 0x00ff00ffu) + 0x00010001u;
  const uint32_t out = ((te >> 8) & 0x00ff00ffu) | (to & 0xff00ff00u);
  /* OVER10: (Cs*255 + Cd*na)/255 = Cs + (Cd*na)/255, then MIN 255 -- a saturating byte add; the
   * alpha byte comes out as a + (255*na)/255 = 255 by itself. OVER00: alpha byte = 255. */
  return sp ? __vaddus4 (out, o) : (out | (0xffu << (8 * AP)));
}

template <int AP>
__device__ __forceinline__ uint4
blend16_packed (uint4 f, const uint4 &o, uint32_t ga, bool sp, bool dp)
{
  constexpr uint32_t AM = 0xffu << (8 * AP);
  /* the four pixels of a vector nearly always share their case: decide once per vector */
  if (ga == 255u && !dp && ((f.x & f.y & f.z & f.w) & AM) == AM) {
    if (((o.x | o.y | o.z | o.w) & AM) == 0u)
      return f;                                       /* transparent all over */
    f.x = blend_px_packed_opaque<AP> (f.x, o.x, sp);
    f.y = blend_px_packed_opaque<AP> (f.y, o.y, sp);
    f.z = blend_px_packed_opaque<AP> (f.z, o.z, sp);
    f.w = blend_px_packed_opaque<AP> (f.w, o.w, sp);
    return f;
  }
  f.x = blend_px_packed<AP> (f.x, o.x, ga, sp, dp);
  f.y = blend_px_packed<AP> (f.y, o.y, ga, sp, dp);
  f.z = blend_px_packed<AP> (f.z, o.z, ga, sp, dp);
  f.w = blend_px_packed<AP> (f.w, o.w, ga, sp, dp);
  return f;
}

/* The scalars of a rectangle that its blend operator takes. PLANE8 has one operator, so its ga
 * and src_premul are constants; a_ga is read by the JF_GA variants only. */
struct RectOp { uint32_t ga, a_ga; bool sp; };

template <int KIND, bool GA>
__device__ __forceinline__ RectOp
rect_op (const RectRef *r)
{
  RectOp op;
  op.ga = KIND == PK_PLANE8 ? 255u : (uint32_t) __ldg (&r->ga);
  op.sp = KIND == PK_PLANE8 ? false : __ldg (&r->src_premul) != 0;
  op.a_ga = GA ? (uint32_t) __ldg (&r->a_ga) : 255u;
  return op;
}

/* One 16-byte vector of frame f blended with one rectangle: oa = its alpha bytes (PLANE8 kinds)
 * or pixel words (packed), oc = its colour bytes (PLANE8 kinds; not read by the packed kinds),
 * dp = destination premultiplied. */
template <int KIND, bool GA>
__device__ __forceinline__ uint4
blend16 (const uint4 &f, uint4 oa, const uint4 &oc, const RectOp &op, bool dp)
{
  if (GA)
    oa = scale16_alpha (oa, op.a_ga);
  if (KIND == PK_PLANE8)
    return blend16_plane8 (f, oa, oc);
  if (KIND == PK_PLANE8_RGB)
    return blend16_rgb24 (f, oa, oc, op.ga, op.sp);
  return blend16_packed<KIND == PK_PACKED_A0 ? 0 : 3> (f, oa, op.ga, op.sp, dp);
}

/* ---------------------------------------------------------------------- */
/* the per-frame blend kernel                                             */

struct RectGeom { int32_t v0, v1, y0, y1; };

__device__ __forceinline__ RectGeom
rect_geom (const RectRef *r)
{
  const int4 g = __ldg (reinterpret_cast<const int4 *> (&r->v0));
  RectGeom o;
  o.v0 = g.x; o.v1 = g.y; o.y0 = g.z; o.y1 = g.w;
  return o;
}

template <int KIND, bool GA = false>
__device__ __forceinline__ uint4
blend_with_rect (uint4 f, const RectRef *r, const RectGeom &g, int v, int y,
    bool dst_premul)
{
  const int32_t pitch = __ldg (&r->pitch);
  const size_t off = (size_t) (y - g.y0) * pitch + (size_t) (v - g.v0) * 16;
  const uint4 oa = ld_overlay16 (ldg_ptr (&r->a) + off);
  const uint4 oc = kind_is_planes (KIND) ? ld_overlay16 (ldg_ptr (&r->c) + off) : oa;
  return blend16<KIND, GA> (f, oa, oc, rect_op<KIND, GA> (r), dst_premul);
}

/* Job fields a CTA keeps in registers while it works through the job. */
struct JobRegs {
  const uint8_t *src;
  uint8_t *dst;
  const RectRef *rects;
  unsigned long long rect_mask;
  int src_pitch, dst_pitch;
  int win_v0, win_y0;
  uint32_t win_nv, total_items, magic;
  int cls, one_rect, flags, row_bytes;
};

__device__ __forceinline__ JobRegs
load_job (const PlaneJob *job)
{
  JobRegs J;
  J.rects = ldg_ptr (&job->rects);
  J.rect_mask = __ldg (&job->rect_mask);
  J.one_rect = __ldg (&job->one_rect);
  J.flags = __ldg (&job->flags);
  J.row_bytes = __ldg (&job->row_bytes);
  J.src = ldg_ptr (&job->src);
  J.dst = ldg_ptr (&job->dst);
  J.src_pitch = __ldg (&job->src_pitch);
  J.dst_pitch = __ldg (&job->dst_pitch);
  J.win_v0 = __ldg (&job->win_v0);
  J.win_nv = (uint32_t) __ldg (&job->win_nv);
  J.win_y0 = __ldg (&job->win_y0);
  J.total_items = J.win_nv * (uint32_t) __ldg (&job->win_rows);
  J.magic = __ldg (&job->div_magic);
  J.cls = __ldg (&job->cls);
  return J;
}

/* Does this 16-byte vector of prepared overlay hold any alpha != 0? PLANE8: an alpha byte
 * per destination byte; packed: the alpha byte of each of the four pixel words. Alpha 0
 * leaves the destination untouched (BLENDSPEC section 2, `continue`), so an in-place blend
 * needs neither read nor write such a vector. */
template <int KIND>
__device__ __forceinline__ bool
any_alpha (const uint4 &oa)
{
  const uint32_t m = oa.x | oa.y | oa.z | oa.w;
  return kind_is_planes (KIND) ? m != 0u : ((m >> (KIND == PK_PACKED_A0 ? 0 : 24)) & 0xffu) != 0u;
}

/* Is every alpha of this vector 255? With ga == 255 that makes asrc = 255, and then all four
 * OVER operators give (255, Cs) whatever the destination holds (its weight 255 - asrc is 0):
 * the destination need not be read. */
template <int KIND>
__device__ __forceinline__ bool
all_opaque (const uint4 &oa)
{
  const uint32_t m = oa.x & oa.y & oa.z & oa.w;
  return kind_is_planes (KIND) ? m == 0xffffffffu : ((m >> (KIND == PK_PACKED_A0 ? 0 : 24)) & 0xffu) == 0xffu;
}

/* One chunk = kItemsPerChunk consecutive 16-byte vectors of one job. A job is
 * a window of one plane whose rows all see the same set of rectangles
 * (rect_mask): the host cuts every plane at the rectangles' top and bottom
 * edges, so the class of a chunk is known before launch and uniform per CTA:
 *   JC_COPY     no rectangle: stream the rows through;
 *   JC_ONE      exactly one rectangle covering the window's whole width:
 *               every vector blends with it, no per-item tests;
 *   JC_ONE_BULK the same, and the rectangle's prepared rows are packed
 *               back to back over exactly the window's columns, so the
 *               chunk's overlay bytes are contiguous: staged through shared
 *               memory by the TMA (group kernel only);
 *   JC_GENERAL  several rectangles and/or partial width: per-item column
 *               tests, rectangles applied in order.
 * Thread t owns items t, t+256, t+512, t+768 of the chunk, so four
 * independent 128-bit frame loads (plus their overlay loads) are in flight
 * per thread before the first is consumed. FAST = 16-byte aligned frame and
 * no ragged vector; otherwise the byte-granular variant runs. LAZY (in-place
 * group launches: dst == src, or host frames blended over PCIe) looks at the
 * overlay first and touches only the vectors it will change: a vector whose
 * alpha is zero everywhere is neither loaded nor stored -- for cues without a
 * background box most of the region never crosses the bus. */
template <int KIND, bool FAST, bool BULK, int LAZY = 0, bool GA = false>
__device__ __forceinline__ void
process_chunk (const JobRegs &J, uint32_t local_chunk)
{
  const uint8_t *src = J.src;
  uint8_t *dst = J.dst;
  const int src_pitch = J.src_pitch, dst_pitch = J.dst_pitch;
  const uint32_t item0 = local_chunk * kItemsPerChunk + threadIdx.x;

  int vv[kUnroll], yy[kUnroll];
  bool act[kUnroll];
#pragma unroll
  for (int k = 0; k < kUnroll; k++) {
    const uint32_t item = item0 + k * kThreads;
    act[k] = item < J.total_items;
    const uint32_t row = J.win_nv == 1u ? item : __umulhi (item, J.magic);
    const uint32_t col = item - row * J.win_nv;
    vv[k] = J.win_v0 + (int) col;
    yy[k] = J.win_y0 + (int) row;
  }

  uint4 f[kUnroll];

  if (FAST) {
    if (J.cls == JC_COPY) {
#pragma unroll
      for (int k = 0; k < kUnroll; k++)
        if (act[k])
          f[k] = ld_frame16 (src + (size_t) yy[k] * src_pitch + (size_t) vv[k] * 16);
#pragma unroll
      for (int k = 0; k < kUnroll; k++)
        if (act[k])
          st_frame16 (dst + (size_t) yy[k] * dst_pitch + (size_t) vv[k] * 16, f[k]);
      return;
    }
    if (BULK && J.cls == JC_ONE_BULK) {
      /* The chunk's slice of the prepared overlay is one contiguous run of
       * bytes (the rectangle spans the window and its rows are packed), so a
       * single thread hands it to the TMA: cp.async.bulk global -> shared,
       * completion on an mbarrier. Meanwhile every thread has its four frame
       * loads in flight; no register holds overlay data while it travels. */
      extern __shared__ __align__ (128) uint8_t ov_smem[];
      __shared__ __align__ (8) unsigned long long ov_bar;
      const RectRef *r = J.rects + J.one_rect;
      const RectGeom g = rect_geom (r);
      const uint32_t first = local_chunk * kItemsPerChunk;
      const uint32_t bytes = min ((uint32_t) kItemsPerChunk, J.total_items - first) * 16u;
      const size_t off = ((size_t) (J.win_y0 - g.y0) * J.win_nv + first) * 16;
      const uint32_t bar = (uint32_t) __cvta_generic_to_shared (&ov_bar);
      const uint32_t sm_a = (uint32_t) __cvta_generic_to_shared (ov_smem);
      if (threadIdx.x == 0) {
        asm volatile ("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r" (bar));
        asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
            :: "r" (bar), "r" (kind_is_planes (KIND) ? 2u * bytes : bytes) : "memory");
        asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
            :: "r" (sm_a), "l" (ldg_ptr (&r->a) + off), "r" (bytes), "r" (bar) : "memory");
        if (kind_is_planes (KIND))
          asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
              :: "r" (sm_a + kItemsPerChunk * 16), "l" (ldg_ptr (&r->c) + off), "r" (bytes), "r" (bar) : "memory");
      }
      if (!LAZY) {
#pragma unroll
        for (int k = 0; k < kUnroll; k++)
          if (act[k])
            f[k] = ld_frame16 (src + (size_t) yy[k] * src_pitch + (size_t) vv[k] * 16);
      }
      __syncthreads ();           /* the barrier is initialised for everybody */
      asm volatile ("{\n"
          ".reg .pred p;\n"
          "OV_WAIT:\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
          "@p bra OV_DONE;\n"
          "bra OV_WAIT;\n"
          "OV_DONE:\n"
          "}" :: "r" (bar) : "memory");
      const RectOp op = rect_op<KIND, GA> (r);
      if (LAZY) {
        /* overlay first. LAZY 1 (in place): only vectors with some alpha are written back, and
         * of those only the ones that are not opaque all over are fetched (all fetches in flight
         * together). LAZY 2 (out of place, a cue with an opaque box): every vector is written,
         * but the ones under an opaque vector are not fetched. Under an opaque vector the
         * result is the overlay colour whatever the frame holds; a stand-in with an opaque
         * alpha byte keeps the packed kinds on their fast path. */
        const bool ga_full = op.ga == 255u;
        const uint32_t fill = KIND == PK_PACKED_A0 ? 0x000000ffu : KIND == PK_PACKED_A3 ? 0xff000000u : 0u;
#pragma unroll
        for (int k = 0; k < kUnroll; k++) {
          uint4 oa = *reinterpret_cast<const uint4 *> (ov_smem + (threadIdx.x + k * kThreads) * 16u);
          if (GA)
            oa = scale16_alpha (oa, op.a_ga);   /* effective alpha: opaque only where a_ga is 255 too */
          if (LAZY == 1)
            act[k] = act[k] && any_alpha<KIND> (oa);
          f[k] = make_uint4 (fill, fill, fill, fill);
          if (act[k] && !(ga_full && all_opaque<KIND> (oa)))
            f[k] = ld_frame16 (src + (size_t) yy[k] * src_pitch + (size_t) vv[k] * 16);
        }
      }
      const bool dp = (J.flags & JF_DST_PREMUL) != 0;
#pragma unroll
      for (int k = 0; k < kUnroll; k++)
        if (act[k]) {
          const uint32_t so = (threadIdx.x + k * kThreads) * 16u;
          const uint4 oa = *reinterpret_cast<const uint4 *> (ov_smem + so);
          const uint4 oc = kind_is_planes (KIND) ? *reinterpret_cast<const uint4 *> (ov_smem + kItemsPerChunk * 16 + so)
              : oa;
          st_frame16 (dst + (size_t) yy[k] * dst_pitch + (size_t) vv[k] * 16,
              blend16<KIND, GA> (f[k], oa, oc, op, dp));
        }
      return;
    }
    /* register-staged variant: table kernel only (the group kernel sends the rare JC_ONE
     * that is not bulk-eligible through the general path and keeps its register budget) */
    if (!BULK && (J.cls == JC_ONE || J.cls == JC_ONE_BULK)) {
      const RectRef *r = J.rects + J.one_rect;
      const RectGeom g = rect_geom (r);
      const int32_t pitch = __ldg (&r->pitch);
      const uint8_t *pa = ldg_ptr (&r->a);
      uint4 oa[kUnroll], oc[kUnroll];
#pragma unroll
      for (int k = 0; k < kUnroll; k++)
        if (act[k])
          f[k] = ld_frame16 (src + (size_t) yy[k] * src_pitch + (size_t) vv[k] * 16);
      /* the rectangle's scalars after the frame loads, out of those loads' live range; the JF_GA
       * alpha is scaled as it arrives, which spills nothing (scaled at the blend, it does) */
      const uint8_t *pc = kind_is_planes (KIND) ? ldg_ptr (&r->c) : pa;
      const RectOp op = rect_op<KIND, GA> (r);
      const bool dp = (J.flags & JF_DST_PREMUL) != 0;
#pragma unroll
      for (int k = 0; k < kUnroll; k++)
        if (act[k]) {
          const size_t off = (size_t) (yy[k] - g.y0) * pitch + (size_t) (vv[k] - g.v0) * 16;
          oa[k] = ld_overlay16 (pa + off);
          oc[k] = kind_is_planes (KIND) ? ld_overlay16 (pc + off) : oa[k];
          if (GA)
            oa[k] = scale16_alpha (oa[k], op.a_ga);
        }
#pragma unroll
      for (int k = 0; k < kUnroll; k++)
        if (act[k])
          /* the packed kinds call their operator directly: through blend16, ptxas makes this
           * table kernel 72 instructions longer and 0.15 % slower on a B200 (config 4) */
          st_frame16 (dst + (size_t) yy[k] * dst_pitch + (size_t) vv[k] * 16,
              kind_is_planes (KIND) ? blend16<KIND, false> (f[k], oa[k], oc[k], op, dp)
              : blend16_packed<KIND == PK_PACKED_A0 ? 0 : 3> (f[k], oa[k], op.ga, op.sp, dp));
      return;
    }
  }

  /* JC_GENERAL, and every class of the byte-granular variant */
  const RectRef *rects = J.rects;
  const unsigned long long mask = J.rect_mask;
  const int flags = J.flags;
  const int row_bytes = J.row_bytes;
  const bool inplace = (flags & JF_INPLACE) != 0;
  const bool dst_premul = (flags & JF_DST_PREMUL) != 0;
  const bool vec_ok = FAST || (flags & JF_VECTOR) != 0;

  /* in place, vectors no rectangle covers are neither read nor written */
  if (inplace) {
    bool hit[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; k++)
      hit[k] = false;
    for (unsigned long long m = mask; m; m &= m - 1) {
      const RectRef *r = rects + (__ffsll ((long long) m) - 1);
      const RectGeom g = rect_geom (r);
      if (LAZY == 1) {
        const int32_t pitch = __ldg (&r->pitch);
        const uint8_t *pa = ldg_ptr (&r->a);
        const uint32_t a_ga = GA ? (uint32_t) __ldg (&r->a_ga) : 255u;
#pragma unroll
        for (int k = 0; k < kUnroll; k++)
          if (act[k] && !hit[k] && vv[k] >= g.v0 && vv[k] < g.v1) {
            uint4 oa = ld_overlay16 (pa + (size_t) (yy[k] - g.y0) * pitch + (size_t) (vv[k] - g.v0) * 16);
            if (GA)
              oa = scale16_alpha (oa, a_ga);
            hit[k] = any_alpha<KIND> (oa);
          }
      } else {
#pragma unroll
        for (int k = 0; k < kUnroll; k++)
          hit[k] = hit[k] || (vv[k] >= g.v0 && vv[k] < g.v1);
      }
    }
#pragma unroll
    for (int k = 0; k < kUnroll; k++)
      act[k] = act[k] && hit[k];
  }

  int nvalid[kUnroll];
#pragma unroll
  for (int k = 0; k < kUnroll; k++) {
    nvalid[k] = FAST ? 16 : min (16, row_bytes - vv[k] * 16);
    if (act[k]) {
      const uint8_t *p = src + (size_t) yy[k] * src_pitch + (size_t) vv[k] * 16;
      if (vec_ok && nvalid[k] == 16)
        f[k] = ld_frame16 (p);
      else
        f[k] = ld_frame_bytes (p, nvalid[k]);
    }
  }

  /* rectangles in blend order; the job's rows are inside every one of them */
  for (unsigned long long m = mask; m; m &= m - 1) {
    const RectRef *r = rects + (__ffsll ((long long) m) - 1);
    const RectGeom g = rect_geom (r);
#pragma unroll
    for (int k = 0; k < kUnroll; k++)
      if (act[k] && vv[k] >= g.v0 && vv[k] < g.v1)
        f[k] = blend_with_rect<KIND, GA> (f[k], r, g, vv[k], yy[k], dst_premul);
  }

#pragma unroll
  for (int k = 0; k < kUnroll; k++) {
    if (act[k]) {
      uint8_t *p = dst + (size_t) yy[k] * dst_pitch + (size_t) vv[k] * 16;
      if (vec_ok && nvalid[k] == 16)
        st_frame16 (p, f[k]);
      else
        st_frame_bytes (p, f[k], nvalid[k]);
    }
  }
}

/* One CTA per chunk (a streaming copy on B200 is fastest as many short-lived
 * CTAs: tools/copybench.cu, DESIGN.md). CTAs do NOT take chunks in list order:
 * the flat chunk list is walked as `lanes` interleaved sequential streams
 *     chunk = (cta % lanes) * per_lane + cta / lanes
 * so that the CTAs resident at any moment are spread over all frames and
 * bands of the launch. Blend chunks (ALU-heavy) and copy chunks (pure HBM
 * streaming) then share every SM all the time and the integer work hides
 * under the memory time, instead of the chip being compute-bound inside the
 * cue bands and idle on the ALUs outside them. */
#ifndef TTMLBLEND_MIN_CTAS
#define TTMLBLEND_MIN_CTAS 5
#endif

/* the chunk of this CTA; lanes_magic = ceil (2^32 / lanes) (chunk_order) */
__device__ __forceinline__ uint32_t
cta_chunk (uint32_t lanes, uint32_t lanes_magic, uint32_t per_lane)
{
  const uint32_t q = lanes == 1u ? blockIdx.x : __umulhi (blockIdx.x, lanes_magic);
  return (blockIdx.x - q * lanes) * per_lane + q;
}

template <int KIND, bool FAST, bool GA = false>
__global__ void __launch_bounds__ (kThreads, FAST ? 4 : 2)
ttmlblend_blend_kernel (const PlaneJob *__restrict__ jobs,
    const uint32_t *__restrict__ chunk_begin, const uint32_t *__restrict__ coarse, int n_jobs,
    uint32_t total_chunks, uint32_t lanes, uint32_t per_lane, uint32_t lanes_magic, int sync)
{
  pdl_begin (sync);
  const uint32_t chunk = cta_chunk (lanes, lanes_magic, per_lane);
  if (chunk >= total_chunks) {
    pdl_end (sync);
    return;
  }

  /* which job: the host's coarse index names the job that holds the first chunk of this
   * chunk's block of kCoarseChunks; from there a short walk over the begins. Every thread does
   * the same (broadcast) loads, so there is no barrier and the cost does not grow with the
   * number of jobs -- a launch may carry the windows of hundreds of frames with different
   * cue layouts. */
  uint32_t j = __ldg (coarse + (chunk >> kCoarseShift));
  while (j + 1u < (uint32_t) n_jobs && __ldg (chunk_begin + j + 1u) <= chunk)
    j++;
  const JobRegs J = load_job (jobs + j);
  process_chunk<KIND, FAST, false, 0, GA> (J, chunk - __ldg (chunk_begin + j));
  pdl_end (sync);
}

/* The job of a band of one frame of a parameter-block launch (group and multi-layout kernels);
 * `rects` is the frame's rectangle table of the band's plane. */
__device__ __forceinline__ JobRegs
band_job (const BandDesc &B, const FramePtrs &F, const RectRef *rects, const int32_t *src_pitch,
    const int32_t *dst_pitch, int flags)
{
  const int pl = B.plane;
  JobRegs J;
  J.src = F.src[pl];
  J.dst = F.dst[pl];
  J.rects = rects;
  J.rect_mask = ((unsigned long long) B.rect_mask_hi << 32) | B.rect_mask_lo;
  J.src_pitch = src_pitch[pl];
  J.dst_pitch = dst_pitch[pl];
  J.win_v0 = B.win_v0;
  J.win_y0 = B.win_y0;
  J.win_nv = (uint32_t) B.win_nv;
  J.total_items = (uint32_t) B.win_nv * (uint32_t) B.win_rows;
  J.magic = B.div_magic;
  J.cls = B.cls;
  J.one_rect = B.one_rect;
  J.flags = flags;
  J.row_bytes = 0;              /* FAST: never read */
  return J;
}

/* The common case -- a batch of frames that share format, size, strides and
 * cue layout (consecutive frames of a stream, or many streams with the same
 * region boxes) -- needs no table in global memory at all: the band list is
 * the same for every frame and only the plane pointers differ, so both fit in
 * the kernel parameters (constant bank). A CTA finds its frame with one
 * multiply, its band with a short scan of uniform compares, and issues its
 * first frame load without a single dependent global load or barrier in
 * front of it (the table search of the generic kernel above costs ~8 % of a
 * streaming copy: tools/copybench.cu "+prologue"). */
template <int KIND, int LAZY, int NF, int NB, bool GA = false>
__global__ void __launch_bounds__ (kThreads, LAZY == 1 ? 4 : TTMLBLEND_MIN_CTAS)
ttmlblend_group_kernel (const __grid_constant__ GroupParamsT<NF, NB> P)
{
  const GroupHeader &Hd = P.h;
  pdl_begin (Hd.flags);
  const uint32_t chunk = cta_chunk (Hd.lanes, Hd.lanes_magic, Hd.per_lane);
  if (chunk >= Hd.total_chunks) {
    pdl_end (Hd.flags);
    return;
  }
  /* ceil (2^32 / 1) does not fit the magic: one chunk per frame is its own case */
  const uint32_t frame = Hd.chunks_per_frame == 1u ? chunk : __umulhi (chunk, Hd.cpf_magic);
  const uint32_t cif = chunk - frame * Hd.chunks_per_frame;
  uint32_t b = 0;
  for (uint32_t i = 1; i < Hd.n_bands; i++)
    b += cif >= P.bands[i].chunk_begin ? 1u : 0u;
  const BandDesc &B = P.bands[b];
  const FramePtrs &F = P.frames[frame];
  const JobRegs J = band_job (B, F, F.rects + Hd.rect_off[B.plane], Hd.src_pitch, Hd.dst_pitch, Hd.flags);
  process_chunk<KIND, true, true, LAZY, GA> (J, cif - B.chunk_begin);
  pdl_end (Hd.flags);
}

/* The same for frames whose band lists differ (many streams, each with its own cue): the
 * distinct band lists sit back to back in the parameters and every frame names the one it
 * uses. A CTA finds its frame by bisecting the frames' first chunks (six uniform
 * constant-bank reads), then its band as above -- still no global load and no barrier before
 * the first frame load. */
template <int KIND, int LAZY, bool GA = false>
__global__ void __launch_bounds__ (kThreads, LAZY == 1 ? 4 : TTMLBLEND_MIN_CTAS)
ttmlblend_multi_kernel (const __grid_constant__ MultiParams P)
{
  pdl_begin (P.flags);
  const uint32_t chunk = cta_chunk (P.lanes, P.lanes_magic, P.per_lane);
  if (chunk >= P.total_chunks) {
    pdl_end (P.flags);
    return;
  }
  uint32_t frame = 0;
#pragma unroll
  for (uint32_t step = kMaxGroupFrames / 2; step > 0; step >>= 1) {
    const uint32_t t = frame + step;
    if (t < P.n_frames && P.frame_begin[t] <= chunk)
      frame = t;
  }
  const uint32_t cif = chunk - P.frame_begin[frame];
  const uint32_t b0 = P.frame_band0[frame], nb = P.frame_nbands[frame];
  uint32_t b = b0;
  for (uint32_t i = 1; i < nb; i++)
    b += cif >= P.bands[b0 + i].chunk_begin ? 1u : 0u;
  const BandDesc &B = P.bands[b];
  const FramePtrs &F = P.frames[frame];
  const JobRegs J = band_job (B, F, F.rects + ((F.pad_ >> (16 * B.plane)) & 0xffffu), P.src_pitch, P.dst_pitch,
      P.flags);
  process_chunk<KIND, true, true, LAZY, GA> (J, cif - B.chunk_begin);
  pdl_end (P.flags);
}

/* The interleaved chunk order of a launch (cta_chunk). Number of lanes: measured on the 4K
 * configs, the packed kinds (more ALU work per blended vector) gain 3 % with 61 lanes, PLANE8
 * loses 2 % against list order, so the default follows the kind; FLUC_TTMLBLEND_LANES overrides
 * both (1 = list order). A prime keeps lane starts from lining up with the frame structure of a
 * batch. */
struct ChunkOrder { uint32_t lanes, per_lane, magic, grid; };

static cudaError_t
chunk_order (int kind, uint32_t total_chunks, ChunkOrder &o)
{
  static int env = -1;
  if (env < 0) {
    const char *e = getenv ("FLUC_TTMLBLEND_LANES");
    env = e ? atoi (e) : 0;
    if (env < 0) env = 0;
    if (env > 4096) env = 4096;
  }
  o.lanes = env ? (uint32_t) env : kind_is_planes (kind) ? 1u : 61u;
  if (total_chunks < o.lanes * 8u)
    o.lanes = 1;
  o.per_lane = (total_chunks + o.lanes - 1) / o.lanes;
  o.grid = o.lanes * o.per_lane;
  /* umulhi (i, ceil (2^32 / lanes)) == i / lanes while i * lanes < 2^32 */
  if ((unsigned long long) o.grid * o.lanes >= (1ull << 32))
    return cudaErrorInvalidValue;
  o.magic = o.lanes == 1 ? 0u : (uint32_t) (((1ull << 32) + o.lanes - 1) / o.lanes);
  return cudaSuccess;
}

template <int V>
using IntC = std::integral_constant<int, V>;

/* Picks the kernel variant of a launch: calls fn (KIND, LAZY, GA), each a std::integral_constant,
 * for its PlaneKind and its JobFlags. LAZY 1: in place (dst == src, host frames over PCIe) under
 * a sparse cue, the overlay is read first and the vectors it would not change are skipped;
 * LAZY 2: out of place, no frame read under opaque vectors. The JF_GA variants exist for the
 * PLANE8 kinds only (the packed kinds apply RectRef::ga in every variant). */
template <typename Fn>
static cudaError_t
with_variant (int kind, int flags, Fn &&fn)
{
  const auto by_look = [&] (auto K) {
    const auto by_ga = [&] (auto L) {
      if constexpr (kind_is_planes (K)) {
        if (flags & JF_GA)
          return fn (K, L, std::true_type ());
      }
      return fn (K, L, std::false_type ());
    };
    return (flags & JF_LAZY) ? by_ga (IntC<1> ()) : (flags & JF_OPAQUE) ? by_ga (IntC<2> ()) : by_ga (IntC<0> ());
  };
  switch (kind) {
    case PK_PLANE8: return by_look (IntC<PK_PLANE8> ());
    case PK_PLANE8_RGB: return by_look (IntC<PK_PLANE8_RGB> ());
    case PK_PACKED_A0: return by_look (IntC<PK_PACKED_A0> ());
    case PK_PACKED_A3: return by_look (IntC<PK_PACKED_A3> ());
    default: return cudaErrorInvalidValue;
  }
}

/* shared memory for the TMA-staged overlay slice of a JC_ONE_BULK chunk */
static size_t
bulk_smem (int kind)
{
  return (kind_is_planes (kind) ? 2 : 1) * kItemsPerChunk * 16;
}

/* One variant of the group kernel: copies what the launch needs into a parameter block of the
 * variant's size (the full-size block itself when NF / NB are the maxima). */
template <int KIND, int LAZY, int NF, int NB, bool GA>
static cudaError_t
launch_group_variant (const GroupParams &P, uint32_t grid, size_t smem, cudaStream_t stream)
{
  const bool pdl = (P.h.flags & JF_PDL) != 0;
  if (NF == kMaxPlainGroupFrames && NB == kMaxGroupBands)
    return launch_ex (ttmlblend_group_kernel<KIND, LAZY, kMaxPlainGroupFrames, kMaxGroupBands, GA>, grid, smem, stream,
        pdl, P);
  GroupParamsT<NF, NB> S;
  S.h = P.h;
  memcpy (S.bands, P.bands, P.h.n_bands * sizeof (BandDesc));
  memcpy (S.frames, P.frames, P.h.n_frames * sizeof (FramePtrs));
  return launch_ex (ttmlblend_group_kernel<KIND, LAZY, NF, NB, GA>, grid, smem, stream, pdl, S);
}

cudaError_t
launch_group (GroupParams &P, int kind, int sync, cudaStream_t stream)
{
  GroupHeader &Hd = P.h;
  Hd.flags = (Hd.flags & ~(JF_PDL | JF_DEP)) | (sync & (JF_PDL | JF_DEP));
  Hd.total_chunks = Hd.n_frames * Hd.chunks_per_frame;
  if (Hd.total_chunks == 0)
    return cudaSuccess;
  ChunkOrder o;
  if (chunk_order (kind, Hd.total_chunks, o) != cudaSuccess)
    return cudaErrorInvalidValue;
  Hd.lanes = o.lanes;
  Hd.per_lane = o.per_lane;
  Hd.lanes_magic = o.magic;
  static const bool compact = !getenv ("FLUC_TTMLBLEND_COMPACT_PARAMS") || atoi (getenv ("FLUC_TTMLBLEND_COMPACT_PARAMS")) != 0;
  return with_variant (kind, Hd.flags, [&] (auto K, auto L, auto G) {
    if (compact && Hd.n_frames <= 4u && Hd.n_bands <= 16u)
      return launch_group_variant<K, L, 4, 16, G> (P, o.grid, bulk_smem (K), stream);
    if (compact && Hd.n_frames <= 32u)
      return launch_group_variant<K, L, 32, kMaxGroupBands, G> (P, o.grid, bulk_smem (K), stream);
    return launch_group_variant<K, L, kMaxPlainGroupFrames, kMaxGroupBands, G> (P, o.grid, bulk_smem (K), stream);
  });
}

cudaError_t
launch_multi (MultiParams &P, int kind, int sync, cudaStream_t stream)
{
  P.flags = (P.flags & ~(JF_PDL | JF_DEP)) | (sync & (JF_PDL | JF_DEP));
  P.total_chunks = P.frame_begin[P.n_frames];
  if (P.total_chunks == 0)
    return cudaSuccess;
  ChunkOrder o;
  if (chunk_order (kind, P.total_chunks, o) != cudaSuccess)
    return cudaErrorInvalidValue;
  P.lanes = o.lanes;
  P.per_lane = o.per_lane;
  P.lanes_magic = o.magic;
  const bool pdl = (P.flags & JF_PDL) != 0;
  return with_variant (kind, P.flags, [&] (auto K, auto L, auto G) {
    return launch_ex (ttmlblend_multi_kernel<K, L, G>, o.grid, bulk_smem (K), stream, pdl, P);
  });
}

cudaError_t
launch_blend (const PlaneJob *d_jobs, const uint32_t *d_chunk_begin, const uint32_t *d_coarse, int n_jobs,
    uint32_t total_chunks, int kind, bool fast, bool ga, int sync, cudaStream_t stream)
{
  if (n_jobs <= 0 || total_chunks == 0)
    return cudaSuccess;
  ChunkOrder o;
  if (chunk_order (kind, total_chunks, o) != cudaSuccess)
    return cudaErrorInvalidValue;
  const bool pdl = (sync & JF_PDL) != 0;
  /* the table kernel has no LAZY variants */
  return with_variant (kind, ga ? JF_GA : 0, [&] (auto K, auto, auto G) {
    return launch_ex (fast ? ttmlblend_blend_kernel<K, true, G> : ttmlblend_blend_kernel<K, false, G>, o.grid, 0,
        stream, pdl, d_jobs, d_chunk_begin, d_coarse, n_jobs, total_chunks, o.lanes, o.per_lane, o.magic, sync);
  });
}

/* ---------------------------------------------------------------------- */
/* once-per-cue overlay prepare                                           */

struct Ayuv { int a, y, u, v; };

/* unpack_BGRA + matrix_prea_rgb_to_yuv / matrix_rgb_to_yuv of video-blend.c */
__device__ __forceinline__ Ayuv
bgra_to_ayuv (uint32_t px, bool premul)
{
  int b = px & 0xff, g = (px >> 8) & 0xff, r = (px >> 16) & 0xff;
  const int a = px >> 24;
  if (premul && a) {
    r = (r * 255 + a / 2) / a;
    g = (g * 255 + a / 2) / a;
    b = (b * 255 + a / 2) / a;
  }
  Ayuv o;
  o.a = a;
  o.y = min (max ((47 * r + 157 * g + 16 * b + 4096) >> 8, 0), 255);
  o.u = min (max ((-26 * r - 87 * g + 112 * b + 32768) >> 8, 0), 255);
  o.v = min (max ((112 * r - 102 * g - 10 * b + 32768) >> 8, 0), 255);
  return o;
}

__device__ __forceinline__ uint32_t
raw_px (const PrepareParams &p, int x, int y)
{
  return *reinterpret_cast<const uint32_t *> (p.raw + (size_t) (y - p.fy) * p.raw_pitch
      + (size_t) (x - p.fx) * 4);
}

/* One prepared element: a pixel (luma, packed), a chroma sample (planar chroma) or a chroma
 * pair (semi-planar chroma), element i of prepared row r. The one definition of the prepare
 * arithmetic for both prepare kernels. */
__device__ __forceinline__ void
prepare_elem (const PrepareParams &p, int i, int r)
{
  const size_t orow = (size_t) r * p.out_pitch;
  const bool premul = p.premul != 0;

  switch (p.mode) {
    case PM_LUMA:{
      const int x = p.v0 * 16 + i, y = p.row0 + r;
      uint8_t a = 0, c = 0;
      if (x >= p.cx0 && x < p.cx1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x, y), premul);
        const int asrc = s.a * p.ga / 255;
        if (asrc) {
          a = (uint8_t) asrc;
          c = (uint8_t) s.y;
        }
      }
      p.out_a[orow + i] = a;
      p.out_c[orow + i] = c;
      break;
    }
    case PM_CHROMA_PLANAR:{
      const int bx = p.v0 * 16 + i, x = p.sub_x * bx, y = p.sub_y * (p.row0 + r);
      uint8_t a = 0, u = 0, v = 0;
      if (x >= p.cx0 && x < p.cx1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x, y), premul);
        const int asrc = s.a * p.ga / 255;
        if (asrc) {
          a = (uint8_t) asrc;
          u = (uint8_t) s.u;
          v = (uint8_t) s.v;
        }
      }
      p.out_a[orow + i] = a;
      p.out_c[orow + i] = u;
      p.out_c2[orow + i] = v;
      break;
    }
    case PM_CHROMA_UV:
    case PM_CHROMA_VU:{
      const int bx = p.v0 * 8 + i, x = p.sub_x * bx, y = p.sub_y * (p.row0 + r);
      uint8_t a = 0, u = 0, v = 0;
      if (x >= p.cx0 && x < p.cx1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x, y), premul);
        const int asrc = s.a * p.ga / 255;
        if (asrc) {
          a = (uint8_t) asrc;
          u = (uint8_t) s.u;
          v = (uint8_t) s.v;
        }
      }
      p.out_a[orow + 2 * i] = a;
      p.out_a[orow + 2 * i + 1] = a;
      p.out_c[orow + 2 * i] = p.mode == PM_CHROMA_UV ? u : v;
      p.out_c[orow + 2 * i + 1] = p.mode == PM_CHROMA_UV ? v : u;
      break;
    }
    case PM_RGB24:
    case PM_BGR24:{
      /* thread = one byte of the row; the colour stays as the source has it (premultiplied or
       * straight: the blend applies the operator that goes with the rectangle's flag) */
      const int byte = p.v0 * 16 + i, x = byte / 3, ch = byte - 3 * x, y = p.row0 + r;
      uint8_t a = 0, c = 0;
      if (x >= p.cx0 && x < p.cx1) {
        const uint32_t px = raw_px (p, x, y);
        const int asrc = (int) (px >> 24) * p.ga / 255;
        if (asrc) {
          a = (uint8_t) asrc;
          const int sh = p.mode == PM_RGB24 ? 16 - 8 * ch : 8 * ch;      /* BGRA word: B 0, G 8, R 16 */
          c = (uint8_t) (px >> sh);
        }
      }
      p.out_a[orow + i] = a;
      p.out_c[orow + i] = c;
      break;
    }
    case PM_V308:
    case PM_IYU2:{
      /* thread = one byte of the row: pixel = byte / 3, channel = byte % 3 */
      const int byte = p.v0 * 16 + i, x = byte / 3, ch = byte - 3 * x, y = p.row0 + r;
      uint8_t a = 0, c = 0;
      if (x >= p.cx0 && x < p.cx1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x, y), premul);
        const int asrc = s.a * p.ga / 255;
        if (asrc) {
          a = (uint8_t) asrc;
          if (p.mode == PM_V308)
            c = (uint8_t) (ch == 0 ? s.y : ch == 1 ? s.u : s.v);
          else
            c = (uint8_t) (ch == 0 ? s.u : ch == 1 ? s.y : s.v);
        }
      }
      p.out_a[orow + i] = a;
      p.out_c[orow + i] = c;
      break;
    }
    case PM_YUY2:
    case PM_UYVY:
    case PM_YVYU:
    case PM_VYUY:{
      /* packed 4:2:2: thread = macropixel; both lumas, chroma from the even pixel */
      const int x0 = 2 * (p.v0 * 4 + i), y = p.row0 + r;
      uint8_t a0 = 0, a1 = 0, y0 = 0, y1 = 0, u = 0, v = 0;
      if (x0 >= p.cx0 && x0 < p.cx1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x0, y), premul);
        const int asrc = s.a * p.ga / 255;
        if (asrc) {
          a0 = (uint8_t) asrc;
          y0 = (uint8_t) s.y;
          u = (uint8_t) s.u;
          v = (uint8_t) s.v;
        }
      }
      if (x0 + 1 >= p.cx0 && x0 + 1 < p.cx1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x0 + 1, y), premul);
        const int asrc = s.a * p.ga / 255;
        if (asrc) {
          a1 = (uint8_t) asrc;
          y1 = (uint8_t) s.y;
        }
      }
      uchar4 al, co;
      if (p.mode == PM_YUY2) {
        al = make_uchar4 (a0, a0, a1, a0);
        co = make_uchar4 (y0, u, y1, v);
      } else if (p.mode == PM_YVYU) {
        al = make_uchar4 (a0, a0, a1, a0);
        co = make_uchar4 (y0, v, y1, u);
      } else if (p.mode == PM_UYVY) {
        al = make_uchar4 (a0, a0, a0, a1);
        co = make_uchar4 (u, y0, v, y1);
      } else {
        al = make_uchar4 (a0, a0, a0, a1);
        co = make_uchar4 (v, y0, u, y1);
      }
      reinterpret_cast<uchar4 *> (p.out_a + orow)[i] = al;
      reinterpret_cast<uchar4 *> (p.out_c + orow)[i] = co;
      break;
    }
    default:{
      const int x = p.v0 * 4 + i, y = p.row0 + r;
      uint32_t w = 0u;
      if (x >= p.cx0 && x < p.cx1) {
        const uint32_t px = raw_px (p, x, y);
        const uint32_t b = px & 0xffu, g = (px >> 8) & 0xffu, rr = (px >> 16) & 0xffu,
            a = px >> 24;
        switch (p.mode) {
          case PM_PACKED_AYUV:{
            const Ayuv s = bgra_to_ayuv (px, premul);
            w = (uint32_t) s.a | ((uint32_t) s.y << 8) | ((uint32_t) s.u << 16) |
                ((uint32_t) s.v << 24);
            break;
          }
          case PM_PACKED_ARGB:
            w = a | (rr << 8) | (g << 16) | (b << 24);
            break;
          case PM_PACKED_ABGR:
            w = a | (b << 8) | (g << 16) | (rr << 24);
            break;
          case PM_PACKED_RGBA:
            w = rr | (g << 8) | (b << 16) | (a << 24);
            break;
          default:             /* PM_PACKED_BGRA */
            w = px;
            break;
        }
        if (a == 0u)
          w = 0u;               /* blends nothing whatever its colour bytes say: keep the word clean */
      }
      reinterpret_cast<uint32_t *> (p.out_a + orow)[i] = w;
      break;
    }
  }
}

/* One thread per prepared element of one rectangle's plane(s). */
__global__ void __launch_bounds__ (256)
ttmlblend_prepare_kernel (const PrepareParams p, int n_elems)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (i >= n_elems || r >= p.rows)
    return;
  prepare_elem (p, i, r);
}

/* Every plane of every rectangle of one overlay_set_positions generation in one launch: a CTA
 * finds its item by bisecting the items' first CTAs (prefix sums of their element counts in
 * whole CTAs, uniform across the CTA), then takes elements row-major inside it. The items sit in
 * the kernel parameters, or in device memory when there are more than fit there. */
__global__ void __launch_bounds__ (256)
ttmlblend_prepare_batch_kernel (const __grid_constant__ PrepareBatch B)
{
  const PrepareItem *items = B.items ? B.items : B.inl;
  const uint32_t cta = blockIdx.x;
  uint32_t lo = 0, hi = B.n_items;            /* the last item whose first CTA is <= cta */
  while (hi - lo > 1) {
    const uint32_t m = (lo + hi) / 2;
    if (items[m].cta0 <= cta)
      lo = m;
    else
      hi = m;
  }
  const PrepareItem &it = items[lo];
  const int64_t e = (int64_t) (cta - it.cta0) * 256 + threadIdx.x;
  const int n = it.n_elems;
  if (e >= (int64_t) n * it.p.rows)
    return;
  const int r = (int) (e / n);
  prepare_elem (it.p, (int) (e - (int64_t) r * n), r);
}

/* NON-PARITY option (fluc_ttmlblend_set_chroma_mode): each 4:2:0 chroma sample takes the
 * alpha-weighted mean colour and the mean alpha of its 2x2 luma pixels instead of the
 * pixel sited at (even x, even y). GStreamer does not do this (BLENDSPEC section 4), so the
 * result is no longer bit-exact with the reference; it removes the chroma fringes the
 * point-sampled siting leaves under anti-aliased glyph edges. One thread per luma column of
 * the 2x2 blocks: it sums its two rows, the horizontal neighbour's sums arrive by warp
 * shuffle, the even lane writes the sample. */
__global__ void __launch_bounds__ (256)
ttmlblend_prepare_chroma_avg_kernel (const PrepareParams p, int n_cols)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;      /* luma column inside the span */
  const int r = blockIdx.y;
  const bool semi = p.mode != PM_CHROMA_PLANAR;
  const int x = 2 * (semi ? p.v0 * 8 : p.v0 * 16) + i;
  int sa = 0, su = 0, sv = 0;
  if (i < n_cols && x >= p.cx0 && x < p.cx1) {
#pragma unroll
    for (int dy = 0; dy < 2; dy++) {
      const int y = 2 * (p.row0 + r) + dy;
      if (y >= p.cy0 && y < p.cy1) {
        const Ayuv s = bgra_to_ayuv (raw_px (p, x, y), p.premul != 0);
        const int asrc = s.a * p.ga / 255;
        sa += asrc;
        su += asrc * s.u;
        sv += asrc * s.v;
      }
    }
  }
  sa += __shfl_xor_sync (0xffffffffu, sa, 1);
  su += __shfl_xor_sync (0xffffffffu, su, 1);
  sv += __shfl_xor_sync (0xffffffffu, sv, 1);
  if ((i & 1) || i >= n_cols)
    return;
  const uint8_t a = (uint8_t) ((sa + 2) >> 2);
  const uint8_t u = sa && a ? (uint8_t) ((su + sa / 2) / sa) : 0;
  const uint8_t v = sa && a ? (uint8_t) ((sv + sa / 2) / sa) : 0;
  const size_t orow = (size_t) r * p.out_pitch;
  const int k = i >> 1;                                      /* chroma sample inside the span */
  if (!semi) {
    p.out_a[orow + k] = a;
    p.out_c[orow + k] = u;
    p.out_c2[orow + k] = v;
  } else {
    p.out_a[orow + 2 * k] = a;
    p.out_a[orow + 2 * k + 1] = a;
    p.out_c[orow + 2 * k] = p.mode == PM_CHROMA_UV ? u : v;
    p.out_c[orow + 2 * k + 1] = p.mode == PM_CHROMA_UV ? v : u;
  }
}

cudaError_t
launch_prepare (const PrepareParams &p, int n_elems, cudaStream_t stream)
{
  if (n_elems <= 0 || p.rows <= 0)
    return cudaSuccess;
  if (p.chroma_average && p.sub_x == 2 && p.sub_y == 2 && p.mode >= PM_CHROMA_PLANAR && p.mode <= PM_CHROMA_VU) {
    for (int r0 = 0; r0 < p.rows; r0 += 65535) {
      PrepareParams q = p;
      const int nr = min (65535, p.rows - r0);
      q.row0 = p.row0 + r0;
      q.rows = nr;
      q.out_a = p.out_a + (size_t) r0 * p.out_pitch;
      q.out_c = p.out_c + (size_t) r0 * p.out_pitch;
      if (p.out_c2) q.out_c2 = p.out_c2 + (size_t) r0 * p.out_pitch;
      dim3 grid ((2 * n_elems + 255) / 256, nr);
      ttmlblend_prepare_chroma_avg_kernel<<<grid, 256, 0, stream>>> (q, 2 * n_elems);
    }
    return cudaGetLastError ();
  }
  const int rows_per_launch = 65535;
  for (int r0 = 0; r0 < p.rows; r0 += rows_per_launch) {
    PrepareParams q = p;
    const int nr = min (rows_per_launch, p.rows - r0);
    q.row0 = p.row0 + r0;
    q.rows = nr;
    q.out_a = p.out_a + (size_t) r0 * p.out_pitch;
    if (p.out_c) q.out_c = p.out_c + (size_t) r0 * p.out_pitch;
    if (p.out_c2) q.out_c2 = p.out_c2 + (size_t) r0 * p.out_pitch;
    dim3 grid ((n_elems + 255) / 256, nr);
    ttmlblend_prepare_kernel<<<grid, 256, 0, stream>>> (q, n_elems);
  }
  return cudaGetLastError ();
}

uint32_t
prepare_batch_plan (PrepareItem *items, uint32_t n)
{
  uint32_t ctas = 0;
  for (uint32_t k = 0; k < n; k++) {
    items[k].cta0 = ctas;
    ctas += (uint32_t) (((uint64_t) items[k].n_elems * (uint64_t) items[k].p.rows + 255) / 256);
  }
  return ctas;
}

cudaError_t
launch_prepare_batch (const PrepareItem *items, uint32_t n, const PrepareItem *d_items, uint32_t ctas,
    cudaStream_t stream)
{
  if (n == 0 || ctas == 0)
    return cudaSuccess;
  PrepareBatch B;
  B.n_items = n;
  B.items = n > kPrepareBatchInline ? d_items : nullptr;
  if (!B.items)
    memcpy (B.inl, items, n * sizeof (PrepareItem));
  ttmlblend_prepare_batch_kernel<<<ctas, 256, 0, stream>>> (B);
  return cudaGetLastError ();
}

/* ---------------------------------------------------------------------- */
/* once per cue: where is the rectangle not transparent?                   */

/* One row's span and group figures: span = (first x, last x) with alpha != 0, or (w, -1); groups =
 * how many of the row's 16-pixel groups hold any alpha != 0, in the low half, and how many are
 * opaque all over (alpha 255), in the high half. Each thread of a 128-thread CTA feeds it pixels
 * x = base + threadIdx.x for base = 0, 128, ... (every lane of a warp at once: the ballots see
 * two 16-pixel groups per warp), 0 past the row's end; rowscan_store reduces and writes it. */
struct RowScan {
  int lo, hi, ng;
};

__device__ __forceinline__ void
rowscan_px (RowScan &s, int x, uint32_t a)
{
  const bool on = a != 0u;
  if (on) {
    s.lo = min (s.lo, x);
    s.hi = max (s.hi, x);
  }
  const uint32_t b = __ballot_sync (0xffffffffu, on);      /* two groups of 16 pixels per warp */
  const uint32_t q = __ballot_sync (0xffffffffu, a == 255u);
  s.ng += ((b & 0xffffu) ? 1 : 0) + ((b >> 16) ? 1 : 0);
  s.ng += (((q & 0xffffu) == 0xffffu) ? 0x10000 : 0) + (((q >> 16) == 0xffffu) ? 0x10000 : 0);
}

/* every thread of the CTA calls it; thread 0 writes */
__device__ __forceinline__ void
rowscan_store (RowScan s, int2 *__restrict__ span, int *__restrict__ groups)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s.lo = min (s.lo, __shfl_xor_sync (0xffffffffu, s.lo, o));
    s.hi = max (s.hi, __shfl_xor_sync (0xffffffffu, s.hi, o));
  }
  __shared__ int s_lo[4], s_hi[4], s_ng[4];
  if ((threadIdx.x & 31) == 0) {
    s_lo[threadIdx.x >> 5] = s.lo;
    s_hi[threadIdx.x >> 5] = s.hi;
    s_ng[threadIdx.x >> 5] = s.ng;      /* the same in every lane of a warp */
  }
  __syncthreads ();
  if (threadIdx.x == 0) {
    *span = make_int2 (min (min (s_lo[0], s_lo[1]), min (s_lo[2], s_lo[3])),
        max (max (s_hi[0], s_hi[1]), max (s_hi[2], s_hi[3])));
    *groups = s_ng[0] + s_ng[1] + s_ng[2] + s_ng[3];
  }
}

/* One CTA per row (RowScan). How sparse / how opaque the cue is decides whether in-place
 * launches look at the overlay before touching the frame. */
__global__ void __launch_bounds__ (128)
ttmlblend_rowspan_kernel (const uint8_t *__restrict__ raw, int pitch, int w, int2 *__restrict__ spans,
    int *__restrict__ groups)
{
  const int y = blockIdx.x;
  const uint32_t *row = reinterpret_cast<const uint32_t *> (raw + (size_t) y * pitch);
  RowScan s = { w, -1, 0 };
  for (int base = 0; base < w; base += blockDim.x) {
    const int x = base + (int) threadIdx.x;
    rowscan_px (s, x, x < w ? row[x] >> 24 : 0u);
  }
  rowscan_store (s, spans + y, groups + y);
}

cudaError_t
launch_rowspan (const uint8_t *raw, int pitch, int w, int h, int2 *spans, int *groups, cudaStream_t stream)
{
  if (w <= 0 || h <= 0)
    return cudaSuccess;
  ttmlblend_rowspan_kernel<<<h, 128, 0, stream>>> (raw, pitch, w, spans, groups);
  return cudaGetLastError ();
}

/* ---------------------------------------------------------------------- */
/* once per cue: region background / opacity composition (pixman 8-bit)    */

/* pixman MUL_UN8: (a * b) / 255, rounded */
__device__ __forceinline__ uint32_t
mul_un8 (uint32_t a, uint32_t b)
{
  const uint32_t t = a * b + 0x80u;
  return ((t >> 8) + t) >> 8;
}

/* premultiplied a8r8g8b8: s OVER d, per channel d = sat (s + d * (255 - s.a) / 255) */
__device__ __forceinline__ uint32_t
over_un8x4 (uint32_t s, uint32_t d)
{
  const uint32_t ia = 255u - (s >> 24);
  uint32_t out = 0u;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint32_t v = ((s >> (8 * k)) & 0xffu) + mul_un8 ((d >> (8 * k)) & 0xffu, ia);
    out |= min (v, 255u) << (8 * k);
  }
  return out;
}

__device__ __forceinline__ uint32_t
in_un8x4 (uint32_t s, uint32_t m)
{
  uint32_t out = 0u;
#pragma unroll
  for (int k = 0; k < 4; k++)
    out |= mul_un8 ((s >> (8 * k)) & 0xffu, m) << (8 * k);
  return out;
}

/* gst_ttmlrender_show_regions without the text rasterisation
 * (/root/reference/plugins/ttml/gstttmlrender.c:1250-1268,1375-1381): opacity 1 draws
 * straight onto the canvas, opacity < 1 goes through a cleared group surface that is then
 * painted with the opacity as mask. One thread per pixel of the (clipped) region box. */
__global__ void __launch_bounds__ (256)
ttmlblend_region_kernel (const RegionParams p)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= p.w || j >= p.h)
    return;
  uint32_t *dst = reinterpret_cast<uint32_t *> (p.canvas + (size_t) (p.y + j) * p.canvas_pitch) + (p.x + i);
  const uint32_t layer = p.layer ?
      *reinterpret_cast<const uint32_t *> (p.layer + (size_t) (p.ly + j) * p.layer_pitch + 4 * (size_t) (p.lx + i)) : 0u;
  uint32_t d = *dst;
  if (p.m8 == 255u) {
    if (p.bg)
      d = over_un8x4 (p.bg, d);
    if (p.layer)
      d = over_un8x4 (layer, d);
  } else {
    uint32_t g = p.bg;                      /* bg OVER cleared group surface */
    if (p.layer)
      g = over_un8x4 (layer, g);
    d = over_un8x4 (in_un8x4 (g, p.m8), d); /* cairo_paint_with_alpha */
  }
  *dst = d;
}

cudaError_t
launch_region (const RegionParams &p, cudaStream_t stream)
{
  if (p.w <= 0 || p.h <= 0)
    return cudaSuccess;
  for (int r0 = 0; r0 < p.h; r0 += 65535) {
    RegionParams q = p;
    q.y = p.y + r0;
    q.ly = p.ly + r0;
    q.h = min (65535, p.h - r0);
    dim3 grid ((p.w + 255) / 256, q.h);
    ttmlblend_region_kernel<<<grid, 256, 0, stream>>> (q);
  }
  return cudaGetLastError ();
}

/* ---------------------------------------------------------------------- */
/* once per cue with a blurred textOutline: pixman-style 2-D convolution   */

/* gst_ttml_blur_image_surface (/root/reference/plugins/ttml/gstttmlblur.c:72-110):
 * a8r8g8b8 source with a (2r+1)^2 kernel of 16.16 fixed-point taps, pixels
 * outside the image are transparent, result = CLIP ((sum + 0x8000) >> 16).
 * 32 x 8 output pixels per CTA; the tile plus its halo and the taps sit in
 * shared memory, one thread per output pixel, four channels per thread. */
constexpr int kBlurTileW = 32, kBlurTileH = 8;

__global__ void __launch_bounds__ (kBlurTileW * kBlurTileH)
ttmlblend_blur_kernel (const uint8_t *__restrict__ src, int w, int h, int src_pitch,
    const int32_t *__restrict__ taps, int radius, uint8_t *__restrict__ dst, int dst_pitch)
{
  extern __shared__ uint32_t blur_smem[];
  const int size = 2 * radius + 1;
  const int tw = kBlurTileW + 2 * radius, th = kBlurTileH + 2 * radius;
  uint32_t *tile = blur_smem;
  int32_t *s_taps = reinterpret_cast<int32_t *> (blur_smem + tw * th);
  const int tid = threadIdx.y * kBlurTileW + threadIdx.x;
  const int x0 = blockIdx.x * kBlurTileW - radius, y0 = blockIdx.y * kBlurTileH - radius;
  for (int i = tid; i < tw * th; i += kBlurTileW * kBlurTileH) {
    const int x = x0 + i % tw, y = y0 + i / tw;
    uint32_t px = 0u;
    if (x >= 0 && x < w && y >= 0 && y < h)
      px = *reinterpret_cast<const uint32_t *> (src + (size_t) y * src_pitch + 4 * (size_t) x);
    tile[i] = px;
  }
  for (int i = tid; i < size * size; i += kBlurTileW * kBlurTileH)
    s_taps[i] = taps[i];
  __syncthreads ();
  const int ox = blockIdx.x * kBlurTileW + threadIdx.x, oy = blockIdx.y * kBlurTileH + threadIdx.y;
  if (ox >= w || oy >= h)
    return;
  int t0 = 0, t1 = 0, t2 = 0, t3 = 0;
  for (int i = 0; i < size; i++) {
    const uint32_t *row = tile + (threadIdx.y + i) * tw + threadIdx.x;
    const int32_t *tr = s_taps + i * size;
    for (int j = 0; j < size; j++) {
      const int32_t f = tr[j];
      const uint32_t px = row[j];
      t0 += (int) (px & 0xffu) * f;
      t1 += (int) ((px >> 8) & 0xffu) * f;
      t2 += (int) ((px >> 16) & 0xffu) * f;
      t3 += (int) (px >> 24) * f;
    }
  }
  t0 = min (max ((t0 + 0x8000) >> 16, 0), 255);
  t1 = min (max ((t1 + 0x8000) >> 16, 0), 255);
  t2 = min (max ((t2 + 0x8000) >> 16, 0), 255);
  t3 = min (max ((t3 + 0x8000) >> 16, 0), 255);
  *reinterpret_cast<uint32_t *> (dst + (size_t) oy * dst_pitch + 4 * (size_t) ox) =
      (uint32_t) t0 | ((uint32_t) t1 << 8) | ((uint32_t) t2 << 16) | ((uint32_t) t3 << 24);
}

cudaError_t
launch_blur (const uint8_t *src, int w, int h, int src_pitch, const int32_t *taps, int radius,
    uint8_t *dst, int dst_pitch, cudaStream_t stream)
{
  if (w <= 0 || h <= 0)
    return cudaSuccess;
  const int size = 2 * radius + 1;
  const size_t smem = ((size_t) (kBlurTileW + 2 * radius) * (kBlurTileH + 2 * radius) +
      (size_t) size * size) * 4;
  if (smem > 200 * 1024)
    return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute (ttmlblend_blur_kernel,
        cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess)
      return e;
  }
  dim3 grid ((w + kBlurTileW - 1) / kBlurTileW, (h + kBlurTileH - 1) / kBlurTileH);
  dim3 block (kBlurTileW, kBlurTileH);
  ttmlblend_blur_kernel<<<grid, block, smem, stream>>> (src, w, h, src_pitch, taps, radius, dst, dst_pitch);
  return cudaGetLastError ();
}

/* ---------------------------------------------------------------------- */
/* Rectangle scaling, once per cue: gst_video_blend_scale_linear_RGBA (docs/BLENDSPEC.md
 * section 10). One thread per destination pixel. Horizontally, ORC's bilinear resample of
 * the two source pixels under 16.16 position x * x_inc with an 8-bit fraction,
 * (a*(256-f) + b*f) >> 8 per byte; vertically, ORC's merge of two such lines,
 * a + (((b-a)*w + 128) >> 8). Which two source rows and which weight a destination row
 * uses comes from the host (`rows`: upstream's two-line cache simulated row by row), so the
 * kernel is stateless. */

__device__ __forceinline__ uint32_t
scale_mix_h (uint32_t a, uint32_t b, uint32_t f)
{
  /* two bytes per multiply: (a & 0x00ff00ff) * (256-f) stays below 2^16 per lane */
  const uint32_t g = 256u - f;
  const uint32_t lo = ((a & 0x00ff00ffu) * g + (b & 0x00ff00ffu) * f) >> 8;
  const uint32_t hi = (((a >> 8) & 0x00ff00ffu) * g + ((b >> 8) & 0x00ff00ffu) * f) >> 8;
  return (lo & 0x00ff00ffu) | ((hi & 0x00ff00ffu) << 8);
}

/* destination pixel x of the row whose source rows and weight are r */
__device__ __forceinline__ uint32_t
scale_px (const uint8_t *__restrict__ src, int src_pitch, int4 r, int x_inc, int x)
{
  const int tmp = x * x_inc;
  const int sx = tmp >> 16;
  const uint32_t f = (uint32_t) (tmp >> 8) & 0xffu;
  const uint32_t *ra = reinterpret_cast<const uint32_t *> (src + (size_t) r.x * src_pitch) + sx;
  const uint32_t *rb = reinterpret_cast<const uint32_t *> (src + (size_t) r.y * src_pitch) + sx;
  const uint32_t a = scale_mix_h (__ldg (ra), __ldg (ra + 1), f);
  const uint32_t b = scale_mix_h (__ldg (rb), __ldg (rb + 1), f);
  uint32_t out = 0;
#pragma unroll
  for (int k = 0; k < 32; k += 8) {
    const int ca = (int) ((a >> k) & 0xffu), cb = (int) ((b >> k) & 0xffu);
    out |= (uint32_t) ((ca + (((cb - ca) * r.z + 128) >> 8)) & 0xff) << k;
  }
  return out;
}

__global__ void __launch_bounds__ (256)
ttmlblend_scale_kernel (const uint8_t *__restrict__ src, int src_pitch, const int4 *__restrict__ rows,
    int x_inc, uint8_t *__restrict__ dst, int dst_pitch, int dw, int dh)
{
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= dw || y >= dh)
    return;
  const int4 r = __ldg (&rows[y]);                /* row a, row b, weight */
  reinterpret_cast<uint32_t *> (dst + (size_t) y * dst_pitch)[x] = scale_px (src, src_pitch, r, x_inc, x);
}

cudaError_t
launch_scale (const uint8_t *src, int src_pitch, const int4 *rows, int x_inc, uint8_t *dst, int dst_pitch,
    int dw, int dh, cudaStream_t stream)
{
  dim3 grid ((unsigned) ((dw + 255) / 256), (unsigned) dh);
  ttmlblend_scale_kernel<<<grid, 256, 0, stream>>> (src, src_pitch, rows, x_inc, dst, dst_pitch, dw, dh);
  return cudaGetLastError ();
}

/* Every rectangle of one overlay_set_render_rectangles call in one launch: one CTA per destination
 * row of every item, which finds its item by bisecting the items' first rows (as
 * ttmlblend_prepare_batch_kernel does). A scaled item's CTA computes its row's pixels from the
 * resident source, stores them and, from the same registers, reduces the row's span and group
 * figures (RowScan) -- the scaled image is not read back for the scan. An item without a row plan
 * only scans its source. Without spans (no auto-crop) nothing is scanned. */
__global__ void __launch_bounds__ (128)
ttmlblend_scale_scan_batch_kernel (const __grid_constant__ ScaleScanBatch B)
{
  const ScaleScanItem *items = B.items ? B.items : B.inl;
  const uint32_t cta = blockIdx.x;
  uint32_t lo = 0, hi = B.n_items;            /* the last item whose first row is <= cta */
  while (hi - lo > 1) {
    const uint32_t m = (lo + hi) / 2;
    if (items[m].row0 <= cta)
      lo = m;
    else
      hi = m;
  }
  const ScaleScanItem &it = items[lo];
  const int y = (int) (cta - it.row0), w = it.w;
  const bool scan = B.spans != nullptr;
  RowScan s = { w, -1, 0 };
  if (it.plan >= 0) {
    const int4 r = __ldg (&B.plans[it.plan + y]);
    uint32_t *out = reinterpret_cast<uint32_t *> (it.dst + (size_t) y * it.dst_pitch);
    for (int base = 0; base < w; base += blockDim.x) {
      const int x = base + (int) threadIdx.x;
      uint32_t px = 0u;
      if (x < w) {
        px = scale_px (it.src, it.src_pitch, r, it.x_inc, x);
        out[x] = px;
      }
      if (scan)
        rowscan_px (s, x, px >> 24);
    }
  } else if (scan) {
    const uint32_t *row = reinterpret_cast<const uint32_t *> (it.src + (size_t) y * it.src_pitch);
    for (int base = 0; base < w; base += blockDim.x) {
      const int x = base + (int) threadIdx.x;
      rowscan_px (s, x, x < w ? row[x] >> 24 : 0u);
    }
  }
  if (scan)
    rowscan_store (s, B.spans + cta, B.groups + cta);
}

uint32_t
scale_scan_batch_plan (ScaleScanItem *items, uint32_t n)
{
  uint32_t rows = 0;
  for (uint32_t k = 0; k < n; k++) {
    items[k].row0 = rows;
    rows += (uint32_t) items[k].h;
  }
  return rows;
}

cudaError_t
launch_scale_scan_batch (const ScaleScanItem *items, uint32_t n, const ScaleScanItem *d_items, const int4 *plans,
    int2 *spans, int *groups, uint32_t rows, cudaStream_t stream)
{
  if (n == 0 || rows == 0)
    return cudaSuccess;
  ScaleScanBatch B;
  B.n_items = n;
  B.items = n > kScaleScanBatchInline ? d_items : nullptr;
  B.plans = plans;
  B.spans = spans;
  B.groups = groups;
  if (!B.items)
    memcpy (B.inl, items, n * sizeof (ScaleScanItem));
  ttmlblend_scale_scan_batch_kernel<<<rows, 128, 0, stream>>> (B);
  return cudaGetLastError ();
}

/* ---------------------------------------------------------------------- */

__global__ void
ttmlblend_scrub_kernel (uint4 *buf, size_t n_vec, uint32_t seed)
{
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t) gridDim.x * blockDim.x;
  for (; i < n_vec; i += stride)
    buf[i] = make_uint4 (seed, (uint32_t) i, seed ^ 0x5a5a5a5au, 0u);
}

cudaError_t
launch_scrub (uint8_t *buf, size_t bytes, cudaStream_t stream)
{
  static uint32_t seed = 1;
  if (bytes < 16)
    return cudaSuccess;
  ttmlblend_scrub_kernel<<<148 * 8, 256, 0, stream>>> (reinterpret_cast<uint4 *> (buf),
      bytes / 16, seed++);
  return cudaGetLastError ();
}

/* bench helper (fluc_ttmlblend_pcie_probe): the zero-copy path's traffic shape with no blend in
 * it -- one CTA per 16 KB, four 128-bit loads per thread in flight, the same bytes written back */
__global__ void __launch_bounds__ (kThreads)
ttmlblend_pcie_probe_kernel (uint8_t *buf, size_t n_vec)
{
  const size_t base = (size_t) blockIdx.x * kItemsPerChunk + threadIdx.x;
  uint4 v[kUnroll];
#pragma unroll
  for (int k = 0; k < kUnroll; k++)
    if (base + (size_t) k * kThreads < n_vec)
      v[k] = ld_frame16 (buf + (base + (size_t) k * kThreads) * 16);
#pragma unroll
  for (int k = 0; k < kUnroll; k++)
    if (base + (size_t) k * kThreads < n_vec) {
      v[k].x ^= 1u;
      st_frame16 (buf + (base + (size_t) k * kThreads) * 16, v[k]);
    }
}

cudaError_t
launch_pcie_probe (uint8_t *buf, size_t bytes, cudaStream_t stream)
{
  const size_t n_vec = bytes / 16;
  if (n_vec == 0)
    return cudaSuccess;
  ttmlblend_pcie_probe_kernel<<<(unsigned) ((n_vec + kItemsPerChunk - 1) / kItemsPerChunk), kThreads, 0, stream>>> (buf, n_vec);
  return cudaGetLastError ();
}

}  // namespace tb
