/*
 * scheduler.cu -- the multi-stream batch scheduler: pending frames -> group launches and table
 * launches, table slots uploaded on a copy stream, batch events / tickets, the linger thread.
 * Shape after the reference's worker-thread-under-a-monitor
 * (/root/reference/libs/flu/downloader/lib/fludownloader.c:490-532).
 */
#include "ttmlblend_internal.h"

namespace tbh {

cudaEvent_t
event_get (Ctx *c)
{
  if (!c->event_pool.empty ()) {
    cudaEvent_t e = c->event_pool.back ();
    c->event_pool.pop_back ();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreateWithFlags (&e, cudaEventDisableTiming | (c->blocking_sync ? cudaEventBlockingSync : 0));
  return e;
}

/* a stream wait captures the event's state when it is enqueued: the event may be recorded again */
StreamAfter::~StreamAfter ()
{
  if (ctx && ev)
    ctx->event_pool.push_back (ev);
}

int
slot_reserve (Ctx *c, TableSlot &s, size_t n, size_t words)
{
  if (s.cap >= n && s.cap_words >= words)
    return 0;
  const size_t cap = std::max<size_t> (256, n * 2), cap_words = std::max<size_t> (4096, words * 2);
  if (s.h_jobs) cudaFreeHost (s.h_jobs);
  if (s.h_begin) cudaFreeHost (s.h_begin);
  if (s.d_jobs) cudaFree (s.d_jobs);
  if (s.d_begin) cudaFree (s.d_begin);
  s.h_jobs = nullptr; s.h_begin = nullptr; s.d_jobs = nullptr; s.d_begin = nullptr;
  s.cap = s.cap_words = 0;
  CU (c, cudaHostAlloc ((void **) &s.h_jobs, cap * sizeof (PlaneJob), cudaHostAllocDefault));
  CU (c, cudaHostAlloc ((void **) &s.h_begin, cap_words * sizeof (uint32_t), cudaHostAllocDefault));
  CU (c, cudaMalloc ((void **) &s.d_jobs, cap * sizeof (PlaneJob)));
  CU (c, cudaMalloc ((void **) &s.d_begin, cap_words * sizeof (uint32_t)));
  if (!s.copied)
    CU (c, cudaEventCreateWithFlags (&s.copied, cudaEventDisableTiming));
  if (!s.uploaded)
    CU (c, cudaEventCreateWithFlags (&s.uploaded, cudaEventDisableTiming));
  s.cap = cap;
  s.cap_words = cap_words;
  return 0;
}

/* Copies `jobs` (one PlaneKind) into a table slot and launches the kernel. The slot's word
 * array holds the first chunk of every job, then the coarse index (job of every
 * 2^kCoarseShift-th chunk) the kernel starts its search from. */
int
launch_jobs (Ctx *c, TableSlot &s, const PlaneJob *jobs, size_t n, int kind, bool fast, int sync)
{
  if (n == 0)
    return 0;
  if (s.copied && s.cap)
    CU (c, cudaEventSynchronize (s.copied));
  uint64_t total64 = 0;
  for (size_t i = 0; i < n; i++)
    total64 += jobs[i].n_chunks;
  if (total64 >= (1ull << 31))
    return FLUC_TTMLBLEND_ERROR_INVALID_ARGUMENT;
  const size_t n_coarse = (size_t) ((total64 + (1u << kCoarseShift) - 1) >> kCoarseShift);
  int rc = slot_reserve (c, s, n, n + n_coarse);
  if (rc)
    return rc;
  uint32_t total = 0;
  uint32_t *coarse = s.h_begin + n;
  size_t next = 0;
  bool ga = false;
  for (size_t i = 0; i < n; i++) {
    ga = ga || (jobs[i].flags & JF_GA);
    s.h_jobs[i] = jobs[i];
    s.h_begin[i] = total;
    total += jobs[i].n_chunks;
    for (; next < n_coarse && ((uint32_t) next << kCoarseShift) < total; next++)
      coarse[next] = (uint32_t) i;
  }
  /* the table goes up on the copy stream, so that it overlaps the kernel still
   * running on the blend stream; the slot is free (its last kernel waited on above) */
  CU (c, cudaMemcpyAsync (s.d_jobs, s.h_jobs, n * sizeof (PlaneJob), cudaMemcpyHostToDevice, c->table_stream));
  CU (c, cudaMemcpyAsync (s.d_begin, s.h_begin, (n + n_coarse) * sizeof (uint32_t), cudaMemcpyHostToDevice,
          c->table_stream));
  CU (c, cudaEventRecord (s.uploaded, c->table_stream));
  CU (c, cudaStreamWaitEvent (c->blend_stream, s.uploaded, 0));
  CU (c, launch_blend (s.d_jobs, s.d_begin, s.d_begin + n, (int) n, total, kind, fast, ga, sync, c->blend_stream));
  CU (c, cudaEventRecord (s.copied, c->blend_stream));    /* slot busy until this kernel is done */
  c->stats.launches++;
  return 0;
}

/* Retires the batches that have finished. Batches complete in launch order (one stream), so
 * the boundary between finished and running ones is found by bisection: a handful of event
 * queries however many batches are in flight, instead of one per batch. */
void
reap_batches (Ctx *c)
{
  size_t n = c->batches.size ();
  if (n == 0)
    return;
  size_t done = 0;              /* batches [0, done) have finished */
  if (cudaEventQuery (c->batches[n - 1].done) == cudaSuccess) {
    done = n;
  } else {
    cudaGetLastError ();
    size_t lo = 0, hi = n - 1;  /* batch hi is running; find the first running one */
    while (lo < hi) {
      const size_t mid = (lo + hi) / 2;
      if (cudaEventQuery (c->batches[mid].done) == cudaSuccess)
        lo = mid + 1;
      else {
        cudaGetLastError ();
        hi = mid;
      }
    }
    done = lo;
  }
  for (size_t i = 0; i < done; i++) {
    Batch &b = c->batches.front ();
    if (b.last_ticket > c->retired_through)
      c->retired_through = b.last_ticket;
    if (b.t0 && b.t1) {
      float ms = 0.f;
      if (cudaEventElapsedTime (&ms, b.t0, b.t1) == cudaSuccess) {
        c->stats.kernel_ms += ms;
        c->stats.kernel_ms_launches++;
      }
      c->timing_pool.push_back (b.t0);
      c->timing_pool.push_back (b.t1);
    }
    c->event_pool.push_back (b.done);
    if (b.ev_in)
      c->event_pool.push_back (b.ev_in);
    if (b.ev_blend)
      c->event_pool.push_back (b.ev_blend);
    if (b.dma && c->dma_outstanding)
      c->dma_outstanding--;
    b.host_ranges.clear ();
    b.keep.clear ();            /* drops the overlay references, keeps the capacity */
    c->keep_pool.push_back (std::move (b.keep));
    c->batches.pop_front ();
  }
  if (c->batches.empty ()) {
    c->inflight_host.clear ();
    /* nothing is running any more: the next launch depends on nothing */
    c->inflight_dst.clear ();
    c->inflight_src.clear ();
  }
}

/* ---- host DMA batches ----------------------------------------------------------------
 * A batch of device-accessible host frames is normally blended zero copy: the kernel reads the
 * rows under the cue over PCIe and writes them back. SM-issued reads are the weak side of that
 * when data flows both ways (36 GB/s each way on one GPU, tools/pcie_ceiling.cu), while the copy
 * engines keep 44-49 GB/s -- but only in big pieces: the 128 row pieces of a 32-frame 4K batch,
 * copied one by one, fall to 29 GB/s. Frames that sit at a constant spacing in host memory
 * (pool frames come in slabs; a pipeline takes them one after the other) turn every piece shape
 * into ONE two-dimensional copy for the whole run: rows under the cue -> full-size device staging
 * frames (copy-in stream), the ordinary group launch blends them there in place (blend stream),
 * rows -> host (copy-out stream); several staging sets (3 for whole batches, 8 for pieces), so
 * copy-in of batch i+1, blend of i and copy-out of i-1 overlap. Taken for a batch iff every frame is such a host frame of one layout
 * that is not "look at the overlay first" (under an opaque box zero copy moves the frame in one
 * direction only, which beats any copy), its windows are (nearly) full rows, and the frames form
 * few enough runs.
 *
 * A batch goes out in pieces of Ctx::dma_piece frames (8), so that the copy-out of one piece overlaps
 * the copy-in of the next inside one call too. Measured, 1 x B200, 32-frame 4K NV12 batches, caller
 * one batch behind: 14.8 k frames/s (42.9 GB/s each way) against 13.2 k zero copy; on two GPUs
 * behind one host bridge 17.65 k against 18.3 k. Which transport wins depends on the box, so the
 * default policy measures (Ctx::DmaChoice, dma_choice_step below); fluc_ttmlblend_set_host_dma /
 * FLUC_TTMLBLEND_HOST_DMA = 0 / 1 force one. profiles/r02_host_dma_notes.md has the history. */
struct DmaRun { size_t first, n; ptrdiff_t spacing; };
struct DmaPlan {
  std::vector<DmaRun> runs;
  std::vector<std::pair<const uint8_t *, uint8_t *>> host_ptrs;   /* per frame and plane, for the copies */
  size_t slot = 0;              /* bytes per device staging frame */
  DmaSet *set = nullptr;
  ptrdiff_t plane_off[3] = { 0, 0, 0 };
  const Layout *layout = nullptr;
  uintptr_t host_lo = 0, host_hi = 0;
};

/* can frames of this layout go through the copy engines at all? */
bool
layout_takes_dma (const Layout *L)
{
  if (!L->grouped || !L->jobs.empty () || (L->gflags & JF_LAZY))
    return false;
  if (L->dma_ok < 0) {
    layout_spans (L, L->spans);
    L->dma_ok = L->spans.empty () ? 0 : 1;
    for (const StageSpan &s : L->spans) {
      const int pitch = L->dst_pitch[s.plane];
      if (s.b0 != 0 || s.nb * 10 < pitch * 9)     /* narrow windows: full rows would move too much */
        L->dma_ok = 0;
    }
  }
  return L->dma_ok == 1;
}

/* does the pending batch qualify? Fills the plan; nothing is changed yet. */
static bool
plan_host_dma (Ctx *c, DmaPlan &plan)
{
  std::vector<PendingFrame> &pf = c->pending;
  if (pf.size () < 4)
    return false;
  const Layout *L = pf[0].layout;
  if (!pf[0].host || !layout_takes_dma (L))
    return false;
  for (int pl = 0; pl < 3; pl++)
    plan.plane_off[pl] = pf[0].dst[pl] ? pf[0].dst[pl] - pf[0].dst[0] : 0;
  size_t hull = 0;
  uintptr_t lo = ~(uintptr_t) 0, hi = 0;
  for (size_t i = 0; i < pf.size (); i++) {
    const PendingFrame &f = pf[i];
    if (!f.host || f.layout->id != L->id || f.layout->windowed != L->windowed)
      return false;
    for (int pl = 0; pl < 3; pl++)
      if ((f.dst[pl] ? f.dst[pl] - f.dst[0] : 0) != plan.plane_off[pl] || f.src[pl] != f.dst[pl])
        return false;
    hull = std::max<size_t> (hull, f.host_hi - f.host_lo);
    lo = std::min (lo, f.host_lo);
    hi = std::max (hi, f.host_hi);
    if (f.host_lo != (uintptr_t) f.dst[0])
      return false;             /* plane 0 first: the device frame mirrors the host frame's layout */
  }
  /* runs of frames at a constant spacing */
  for (size_t i = 0; i < pf.size ();) {
    DmaRun r = { i, 1, 0 };
    if (i + 1 < pf.size ()) {
      r.spacing = pf[i + 1].dst[0] - pf[i].dst[0];
      if (r.spacing >= (ptrdiff_t) hull)
        while (r.first + r.n < pf.size () && pf[r.first + r.n].dst[0] - pf[r.first + r.n - 1].dst[0] == r.spacing)
          r.n++;
    }
    plan.runs.push_back (r);
    i += r.n;
  }
  if (plan.runs.size () * L->spans.size () > 48 || plan.runs.size () * 3 > pf.size ())
    return false;               /* too many copies for what they move: zero copy it is */
  plan.slot = align_up (hull, 256);
  plan.layout = L;
  plan.host_lo = lo;
  plan.host_hi = hi;
  return true;
}

/* the batch goes through the copy engines: a staging set, and the frames point into it */
static bool
commit_host_dma (Ctx *c, DmaPlan &plan)
{
  std::vector<PendingFrame> &pf = c->pending;
  /* a staging set (its previous copy-out is waited for on the copy-in stream, not here) */
  DmaSet &set = c->dma_sets[c->next_dma_set];
  const size_t need = plan.slot * pf.size ();
  if (set.bytes < need) {
    if (set.used && cudaEventSynchronize (set.done) != cudaSuccess)
      return false;
    if (set.dev)
      cudaFree (set.dev);
    set.dev = nullptr;
    set.bytes = 0;
    if (cudaMalloc ((void **) &set.dev, need) != cudaSuccess) {
      cudaGetLastError ();
      return false;
    }
    set.bytes = need;
    c->dma_choice.cold = true;
  }
  c->next_dma_set = (c->next_dma_set + 1) % (c->dma_piece ? kDmaSets : 3);
  plan.set = &set;
  /* from here on the frames are blended where the copies put them */
  plan.host_ptrs.resize (pf.size ());
  for (size_t i = 0; i < pf.size (); i++) {
    plan.host_ptrs[i] = { pf[i].src[0], pf[i].dst[0] };
    uint8_t *dev = set.dev + i * plan.slot;
    for (int pl = 0; pl < 3; pl++)
      if (pf[i].dst[pl]) {
        pf[i].dst[pl] = dev + plan.plane_off[pl];
        pf[i].src[pl] = pf[i].dst[pl];
      }
  }
  return true;
}

/* the 2-D copies of a DMA batch, one per run and span: a span's rows are contiguous (full rows) */
static int
dma_copies (Ctx *c, const DmaPlan &plan, bool in)
{
  const Layout *L = plan.layout;
  for (const DmaRun &r : plan.runs)
    for (const StageSpan &s : L->spans) {
      const size_t pitch = (size_t) L->dst_pitch[s.plane];
      const size_t off = (size_t) plan.plane_off[s.plane] + (size_t) s.y0 * pitch;
      const size_t width = (size_t) (s.rows - 1) * pitch + (size_t) s.nb;
      uint8_t *host = plan.host_ptrs[r.first].second + off;
      uint8_t *dev = plan.set->dev + r.first * plan.slot + off;
      const size_t hp = r.n > 1 ? (size_t) r.spacing : width, dp = plan.slot;
      if (in)
        CU (c, cudaMemcpy2DAsync (dev, dp, host, hp, width, r.n, cudaMemcpyHostToDevice, c->dma_in));
      else
        CU (c, cudaMemcpy2DAsync (host, hp, dev, dp, width, r.n, cudaMemcpyDeviceToHost, c->dma_out));
    }
  return 0;
}

/* The measured choice between the two transports (Ctx::DmaChoice), after a qualifying batch of n
 * frames went out; its completion is recorded on `done_stream`. */
static void
dma_choice_step (Ctx *c, size_t n, bool was_dma, cudaStream_t done_stream)
{
  Ctx::DmaChoice &d = c->dma_choice;
  if (!d.ev[0][0])
    for (auto &pair : d.ev)
      for (cudaEvent_t &e : pair)
        if (cudaEventCreate (&e) != cudaSuccess) {
          cudaGetLastError ();
          c->host_dma_policy = 0;       /* no events, no measurement: zero copy */
          return;
        }
  if (!d.judged && d.ended[0] && d.ended[1]) {
    if (cudaEventQuery (d.ev[0][1]) == cudaSuccess && cudaEventQuery (d.ev[1][1]) == cudaSuccess) {
      float ms[2] = { 0.f, 0.f };
      if (cudaEventElapsedTime (&ms[0], d.ev[0][0], d.ev[0][1]) == cudaSuccess &&
          cudaEventElapsedTime (&ms[1], d.ev[1][0], d.ev[1][1]) == cudaSuccess && ms[0] > 0.f && ms[1] > 0.f) {
        d.rate[0] = d.frames[0] / ms[0];
        d.rate[1] = d.frames[1] / ms[1];
        d.dma = d.rate[0] > d.rate[1] * 1.02f;
        TBLOG (1, "host frames: copy engines %.2f frames/ms, zero copy %.2f frames/ms over %u / %u frames: %s from here on",
            d.rate[0], d.rate[1], d.frames[0], d.frames[1], d.dma ? "copy engines" : "zero copy");
      }
      d.judged = true;
      d.trials++;
    }
    cudaGetLastError ();        /* not ready is not an error */
  }
  if (d.phase < 2) {
    const int m = d.phase;
    if (m == 0 && !was_dma) {
      /* the copy engines were wanted and not had (no memory for a staging set): zero copy, try later */
      d.phase = 2;
      d.dma = false;
      d.judged = true;
      d.left = kDmaSteadyFrames;
      return;
    }
    if (m == 0 && d.cold) {
      d.cold = false;
      d.begun[0] = false;       /* an allocation in the middle: the trial starts over with the next batch */
      return;
    }
    /* a trial times the bus, not the caller: a pause in the middle (several batch times) voids it,
     * and a caller that keeps pausing is not bound by the bus -- zero copy, look again later */
    const auto now = std::chrono::steady_clock::now ();
    const bool paused = d.begun[m] && now - d.last > std::chrono::milliseconds (20);
    d.last = now;
    if (paused) {
      d.begun[m] = false;
      if (++d.gaps >= 8) {
        d.gaps = 0;
        d.phase = 2;
        d.dma = false;
        d.judged = true;
        d.left = 2048;
        return;
      }
    }
    if (!d.begun[m]) {
      /* the trial is timed from the completion of its first batch */
      if (cudaEventRecord (d.ev[m][0], done_stream) != cudaSuccess)
        cudaGetLastError ();
      d.begun[m] = true;
      d.frames[m] = 0;
      d.left = kDmaTrialFrames;
      return;
    }
    d.frames[m] += (uint32_t) n;
    d.left -= (int64_t) n;
    if (d.left <= 0) {
      if (cudaEventRecord (d.ev[m][1], done_stream) != cudaSuccess)
        cudaGetLastError ();
      d.ended[m] = true;
      d.phase++;
      if (d.phase == 2) {
        d.left = d.trials == 0 ? 2048 : d.trials == 1 ? 8192 : kDmaSteadyFrames;
        d.judged = false;
      }
    }
    return;
  }
  d.left -= (int64_t) n;
  if (d.left <= 0 && d.judged) {
    d.phase = 0;
    d.begun[0] = d.begun[1] = d.ended[0] = d.ended[1] = false;
  }
}

/* Launches everything pending as one batch (per plane kind). mu held. */
int
launch_pending (Ctx *c)
{
  if (c->pending.empty ())
    return 0;
  NvtxRange nvtx ("ttmlblend.launch_batch");
  /* finished batches are retired in bulk: an event query per launch would be a fifth of the cost
   * of a one-frame launch (wait / sync / stats retire them too) */
  if (c->batches.size () >= 32)
    reap_batches (c);
  DmaPlan plan;
  const bool qualifies = c->host_dma_policy != 0 && plan_host_dma (c, plan);
  const bool dma = qualifies && c->dma_now () && commit_host_dma (c, plan);
  const size_t n_frames = c->pending.size ();
  Batch b = {};
  b.last_ticket = c->pending.back ().ticket;
  b.dma = dma;
  if (!c->keep_pool.empty ()) {
    b.keep = std::move (c->keep_pool.back ());
    c->keep_pool.pop_back ();
  }
  std::vector<PlaneJob> *by_kind = c->by_kind;        /* PlaneKind x {byte-granular, fast}; scratch */
  for (int k = 0; k < kPlaneKinds * 2; k++)
    by_kind[k].clear ();
  std::vector<Group> &groups = c->groups;
  groups.clear ();
  size_t n_multis = 0;
  std::vector<int> &frame_group = c->frame_group;
  frame_group.assign (c->pending.size (), -1);
  size_t fi = 0;
  for (PendingFrame &f : c->pending) {
    emit_table_jobs (f.layout->jobs, f, by_kind);
    if (f.layout->grouped) {
      int gi = -1;
      for (size_t k = 0; k < groups.size (); k++)
        if (group_accepts (groups[k], f)) {
          gi = (int) k;
          break;
        }
      if (gi < 0) {
        groups.emplace_back ();
        gi = (int) groups.size () - 1;
        group_start (groups[gi], f);
      }
      group_add (groups[gi], f);
      frame_group[fi] = gi;
    }
    fi++;
    if (f.host)
      b.host_ranges.add (f.host_lo, f.host_hi);
    if (f.overlay && (b.keep.empty () || b.keep.back () != f.overlay))
      b.keep.push_back (f.overlay);     /* consecutive frames of one cue: one reference */
    if (f.prep && !f.prep->blend_waited) {
      /* once per prepared overlay: later launches follow in stream order */
      f.prep->blend_waited = true;
      CU (c, cudaStreamWaitEvent (c->blend_stream, f.prep->ready, 0));
      c->blend_stream_waits = true;
    }
    if (f.after && !f.after->resolved) {
      /* the caller's work before submit_many_after: once per call; when it has already finished,
       * no wait, and the launch keeps programmatic dependent launch */
      f.after->resolved = true;
      const cudaError_t q = cudaEventQuery (f.after->ev);
      if (q != cudaSuccess) {
        if (q != cudaErrorNotReady)
          CU (c, q);
        cudaGetLastError ();
        CU (c, cudaStreamWaitEvent (c->blend_stream, f.after->ev, 0));
        c->blend_stream_waits = true;
      }
    }
    c->stats.frames_blended++;
    c->stats.algorithmic_bytes += f.layout->algo_bytes;
  }
  /* Many streams with different cue layouts give many groups of a frame or two, and a launch
   * of a few hundred chunks leaves most of the chip idle (tools/many_cues_probe.py: 61 group
   * launches for 256 1080p frames ran at half the rate of 4). Small groups are dissolved --
   * when that saves a launch, i.e. there are at least two of them or a table launch of
   * whole-vector windows is going out anyway. */
  {
    size_t n_small = 0, n_table = 0;
    for (int k = 1; k < kPlaneKinds * 2; k += 2)
      n_table += by_kind[k].size ();
    for (Group &g : groups) {
      g.dissolved = (uint64_t) g.P.h.n_frames * g.P.h.chunks_per_frame < (uint64_t) kMinGroupChunks;
      n_small += g.dissolved ? 1 : 0;
    }
    if (n_small < 2 && n_table == 0)
      for (Group &g : groups)
        g.dissolved = false;
    /* their frames are packed into multi-layout launches (band lists in the parameters,
     * up to 64 frames and kMaxMultiBands bands each); what does not fit goes to the table */
    fi = 0;
    for (PendingFrame &f : c->pending) {
      const int gi = frame_group[fi++];
      if (gi < 0 || !groups[gi].dissolved)
        continue;
      bool placed = false;
      if (c->use_multi) {
        for (size_t k = 0; k < n_multis && !placed; k++)
          placed = multi_add (*c->multis[k], f);
        if (!placed) {
          if (n_multis == c->multis.size ())
            c->multis.emplace_back (new MultiGroup ());
          multi_start (*c->multis[n_multis], f);
          placed = multi_add (*c->multis[n_multis], f);
          n_multis += placed ? 1 : 0;
        }
      }
      if (!placed)
        emit_table_jobs (f.layout->gjobs, f, by_kind);
    }
  }
  const uint64_t first_ticket = c->pending.front ().ticket;
  /* Programmatic dependent launch: a launch may start while earlier ones still run. That is
   * only right for frames that do not touch what those read or write: the ranges of every
   * batch launched since the last dependent one are remembered, and a batch that writes into
   * them, or reads what they write, has its first launch wait for everything before it
   * (JF_DEP); after such a launch only its own ranges can still be in flight. */
  int sync = 0;
  if (c->use_pdl) {
    const bool timed = c->profiling && (c->profile_seq % c->profile_every) == 0;
    bool dep = c->inflight_dst.v.size () + c->inflight_src.v.size () > 4096 || timed || c->isolate_next;
    c->isolate_next = timed;    /* an event pair measures one launch alone: neither it nor its successor overlaps */
    if (!dep)
      dep = sets_overlap (c->pending_dst, c->inflight_dst) || sets_overlap (c->pending_dst, c->inflight_src) ||
          sets_overlap (c->pending_src, c->inflight_dst);
    /* Behind a stream wait (a new cue's prepare, the copies of a DMA batch) the
     * launch goes out as an ordinary one: a programmatic launch behind a stream wait holds back
     * the completion of what was recorded before the wait (measured: the copy-out gated by an
     * event after kernel i did not start until the copy-in kernel i+1 waits for had finished).
     * An ordinary launch is ordered after everything before it, like a dependent one. */
    const bool behind_wait = c->blend_stream_waits || dma || c->dma_outstanding;
    c->blend_stream_waits = false;
    if (dep || behind_wait) {
      c->inflight_dst.clear ();
      c->inflight_src.clear ();
      if (dep && !behind_wait)
        c->stats.dependent_launches++;
    }
    c->inflight_dst.merge (c->pending_dst);
    c->inflight_src.merge (c->pending_src);
    sync = behind_wait ? 0 : JF_PDL | (dep ? JF_DEP : 0);
  }
  c->pending.clear ();
  c->pending_dst.clear ();
  c->pending_src.clear ();
  size_t n_launches = n_multis;
  for (Group &g : groups)
    n_launches += g.dissolved ? 0 : 1;
  for (int k = 0; k < kPlaneKinds * 2; k++)
    n_launches += !by_kind[k].empty ();
  /* From here on the frames are no longer queued: whatever happens, a batch with a `done` event
   * is pushed, so that wait() on these tickets synchronises with what did get launched, and a
   * failure half way (out of memory for a table slot, say -- the context stays usable) is
   * remembered for them instead of being reported as finished work. */
  auto issue = [&]() -> int {
    /* an event pair keeps the batch from overlapping its neighbours (~2 us of stream time):
     * sample every profile_every-th batch. A batch of several launches (several groups /
     * kinds) is timed from before its first to after its last launch. */
    if (c->profiling && n_launches >= 1 && (c->profile_seq++ % c->profile_every) == 0) {
      for (cudaEvent_t *e : { &b.t0, &b.t1 }) {
        if (!c->timing_pool.empty ()) {
          *e = c->timing_pool.back ();
          c->timing_pool.pop_back ();
        } else {
          CU (c, cudaEventCreate (e));
        }
      }
    }
    if (dma) {
      /* copy-in: after the staging set's previous copy-out, and after the newest batch still in
       * flight that touches the same host frames (its copy-out / its zero-copy kernel) */
      if (plan.set->used)
        CU (c, cudaStreamWaitEvent (c->dma_in, plan.set->done, 0));
      int waited_on = -1, back = 0;
      for (auto it = c->batches.rbegin (); it != c->batches.rend (); ++it, ++back)
        if (sets_overlap (it->host_ranges, b.host_ranges)) {
          CU (c, cudaStreamWaitEvent (c->dma_in, it->done, 0));
          waited_on = back;
          break;
        }
      TBLOG (2, "dma batch: %zu frames, %zu run(s) x %zu span(s), %zu host range(s), %zu batches in flight, copy-in waits for batch -%d",
          frame_group.size (), plan.runs.size (), plan.layout->spans.size (), b.host_ranges.v.size (), c->batches.size (),
          waited_on + 1);
      static const bool trace = getenv ("FLUC_TTMLBLEND_DMA_TRACE") != nullptr;
      cudaEvent_t tr[4] = { nullptr, nullptr, nullptr, nullptr };
      if (trace) {
        for (auto &e : tr)
          cudaEventCreate (&e);
        cudaEventRecord (tr[0], c->dma_in);
      }
      int rc = dma_copies (c, plan, true);
      if (rc)
        return rc;
      if (trace) {
        cudaEventRecord (tr[1], c->dma_in);
        c->dma_trace.push_back ({ tr[0], tr[1], tr[2], tr[3] });
      }
      /* events of its own for every hand-over between the three streams, kept until the batch is
       * retired: an event that is recorded again on another stream while a wait on its earlier
       * record is still queued is not something to lean on */
      b.ev_in = event_get (c);
      CU (c, cudaEventRecord (b.ev_in, c->dma_in));
      CU (c, cudaStreamWaitEvent (c->blend_stream, b.ev_in, 0));
      c->stats.host_dma_batches++;
    } else if (c->dma_outstanding) {
      /* zero-copy or device frames after DMA batches: batches complete in launch order (wait and
       * the bulk retirement rely on it), and a zero-copy frame may be one a copy-out still writes */
      for (auto it = c->batches.rbegin (); it != c->batches.rend (); ++it)
        if (it->dma) {
          CU (c, cudaStreamWaitEvent (c->blend_stream, it->done, 0));
          break;
        }
    }
    if (b.t0)
      CU (c, cudaEventRecord (b.t0, c->blend_stream));
    for (Group &g : groups) {
      if (g.dissolved)
        continue;
      CU (c, launch_group (g.P, g.kind, sync, c->blend_stream));
      sync &= ~JF_DEP;          /* the launches of one batch are independent of each other */
      c->stats.launches++;
      c->stats.group_launches++;
      if (g.P.h.flags & JF_LAZY)
        c->stats.lazy_launches++;
      if (g.P.h.flags & JF_OPAQUE)
        c->stats.opaque_skip_launches++;
    }
    for (size_t k = 0; k < n_multis; k++) {
      MultiGroup &m = *c->multis[k];
      CU (c, launch_multi (m.P, m.kind, sync, c->blend_stream));
      sync &= ~JF_DEP;
      c->stats.launches++;
      c->stats.multi_launches++;
      if (m.P.flags & JF_LAZY)
        c->stats.lazy_launches++;
      if (m.P.flags & JF_OPAQUE)
        c->stats.opaque_skip_launches++;
    }
    for (int k = 0; k < kPlaneKinds * 2; k++) {
      if (by_kind[k].empty ())
        continue;
      TableSlot &s = c->slots[c->next_slot];
      c->next_slot = (c->next_slot + 1) % kTableSlots;
      int rc = launch_jobs (c, s, by_kind[k].data (), by_kind[k].size (), k / 2, (k & 1) != 0, sync);
      if (rc)
        return rc;
      sync &= ~JF_DEP;
    }
    if (b.t1)
      CU (c, cudaEventRecord (b.t1, c->blend_stream));
    if (dma) {
      b.ev_blend = event_get (c);
      CU (c, cudaEventRecord (b.ev_blend, c->blend_stream));
      CU (c, cudaStreamWaitEvent (c->dma_out, b.ev_blend, 0));
      if (!c->dma_trace.empty () && c->dma_trace.back ()[2])
        cudaEventRecord (c->dma_trace.back ()[2], c->dma_out);
      int rc = dma_copies (c, plan, false);
      if (rc)
        return rc;
      if (!c->dma_trace.empty () && c->dma_trace.back ()[3])
        cudaEventRecord (c->dma_trace.back ()[3], c->dma_out);
      CU (c, cudaEventRecord (plan.set->done, c->dma_out));
      plan.set->used = true;
    }
    return 0;
  };
  const int rc = issue ();
  if (rc) {
    if (c->failed_ranges.size () >= 64)
      c->failed_ranges.pop_front ();
    c->failed_ranges.push_back ({ first_ticket, b.last_ticket, rc });
    if (b.t0) { c->timing_pool.push_back (b.t0); b.t0 = nullptr; }
    if (b.t1) { c->timing_pool.push_back (b.t1); b.t1 = nullptr; }
  }
  b.done = event_get (c);
  if (b.done && cudaEventRecord (b.done, dma ? c->dma_out : c->blend_stream) == cudaSuccess) {
    if (dma)
      c->dma_outstanding++;
    c->batches.push_back (std::move (b));
    if (qualifies && c->host_dma_policy == 2)
      dma_choice_step (c, n_frames, dma, dma ? c->dma_out : c->blend_stream);
  } else {
    /* not even an event: only a broken context gets here */
    cudaGetLastError ();
    if (b.done)
      c->event_pool.push_back (b.done);
    if (!c->sticky) {
      c->sticky = FLUC_TTMLBLEND_ERROR_CUDA;
      c->cuda_error = "launch_pending: cannot record the batch event";
    }
  }
  c->launched_cv.notify_all ();
  return rc ? rc : c->sticky;
}

void
scheduler_main (Ctx *c)
{
  cudaSetDevice (c->device);
  std::unique_lock<std::mutex> lk (c->mu);
  while (!c->quit) {
    if (c->pending.empty () || c->linger_us == 0) {
      c->cv.wait (lk);
      continue;
    }
    const auto deadline = c->oldest_pending + std::chrono::microseconds (c->linger_us);
    if (std::chrono::steady_clock::now () >= deadline) {
      if (!c->sticky)
        launch_pending (c);
      else {
        c->pending.clear ();
        c->pending_dst.clear ();
        c->pending_src.clear ();
      }
      c->launched_cv.notify_all ();   /* also when the launch failed: waiters must not sleep on */
    } else {
      c->cv.wait_until (lk, deadline);
    }
  }
}

}  // namespace tbh
