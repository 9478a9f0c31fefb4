// tools/e2e_multi.cc -- the host-frame path (fluc_ttmlblend_blend_host_many, pinned pool frames,
// config 3: 4K NV12, two full-width translucent regions, 32 frames per call) on SEVERAL GPUs at
// once, through the C ABI only, with no Python / torch in the process: G workers, one per GPU,
// as G processes (fork before CUDA) or as G threads of one process. Scratch measurement beside
// tools/pcie_ceiling.cu: the same box, the same moment, ceiling and product path side by side.
//
//   build/e2e_multi --gpus 0,1,2,3 [--threads] [--secs 2] [--pin] [--opaque]
//   (FLUC_TTMLBLEND_SYNC=block selects blocking waits in the library)
#include "../include/fluc_ttmlblend.h"

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <sched.h>
#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

static double
now ()
{
  return std::chrono::duration<double> (std::chrono::steady_clock::now ().time_since_epoch ()).count ();
}

constexpr int kMaxGpus = 16;
struct Shared {
  std::atomic<int> arrived, generation, failed;
  double fps[kMaxGpus], gbs[kMaxGpus];
};

static void
barrier (Shared *sh, int n)
{
  const int gen = sh->generation.load ();
  if (sh->arrived.fetch_add (1) + 1 == n) {
    sh->arrived.store (0);
    sh->generation.fetch_add (1);
  } else {
    while (sh->generation.load () == gen && !sh->failed.load ())
      sched_yield ();
  }
}

struct Options {
  std::vector<int> gpus;
  bool threads = false, pin = false, opaque = false, pageable = false;
  double secs = 2.0;
  int batch = 32;
  int depth = 1;                /* batches handed over before the oldest one is waited for */
};

#define OK(x) do { int rc_ = (x); if (rc_) { fprintf (stderr, "%s: %s\n", #x, fluc_ttmlblend_strerror (rc_)); _exit (3); } } while (0)

static void
worker (const Options &o, int w, Shared *sh)
{
  const int G = (int) o.gpus.size ();
  if (o.pin) {
    cpu_set_t all, mine;
    CPU_ZERO (&mine);
    if (sched_getaffinity (0, sizeof all, &all) == 0) {
      std::vector<int> cpus;
      for (int i = 0; i < CPU_SETSIZE; i++)
        if (CPU_ISSET (i, &all))
          cpus.push_back (i);
      const size_t per = std::max<size_t> (1, cpus.size () / G);
      for (size_t i = w * per; i < std::min (cpus.size (), (w + 1) * per); i++)
        CPU_SET (cpus[i], &mine);
      if (CPU_COUNT (&mine))
        sched_setaffinity (0, sizeof mine, &mine);
    }
  }
  const int W = 3840, H = 2160;
  FlucTtmlBlend *ctx = nullptr;
  OK (fluc_ttmlblend_new (o.gpus[w], &ctx));
  /* ttmlrender's frame-sized premultiplied BGRA image: two full-width boxes, black at 75 %
   * (or opaque), with brighter stripes standing in for text */
  std::vector<uint8_t> img ((size_t) W * H * 4, 0);
  const FlucTtmlBlendRect regions[2] = { { 0, 1728, W, 360 }, { 0, 72, W, 144 } };
  for (const FlucTtmlBlendRect &r : regions)
    for (int y = r.y; y < r.y + r.h; y++)
      for (int x = 0; x < W; x++) {
        uint8_t *p = &img[((size_t) y * W + x) * 4];
        const bool text = ((x / 24) & 1) && ((y / 12) % 3 == 1);
        const uint8_t a = o.opaque || text ? 255 : 191;
        const uint8_t c = text ? 255 : 0;
        p[0] = p[1] = p[2] = c;
        p[3] = a;
      }
  OK (fluc_ttmlblend_overlay_set (ctx, 1, img.data (), W, H, W * 4, regions, 2));
  OK (fluc_ttmlblend_set_batch (ctx, (uint32_t) o.batch, 0));
  std::vector<FlucTtmlBlendFrame> sets[8];
  const int n_sets = o.depth + 1;
  std::vector<uint32_t> streams ((size_t) o.batch, 1u);
  for (int si = 0; si < n_sets; si++) {
    auto &set = sets[si];
    set.resize ((size_t) o.batch);
    for (auto &f : set) {
      if (o.pageable) {         /* ordinary memory, GStreamer's default NV12 layout */
        uint8_t *m = (uint8_t *) malloc ((size_t) W * H * 3 / 2);
        f.plane[0] = m;
        f.plane[1] = m + (size_t) W * H;
        f.stride[0] = f.stride[1] = W;
      } else {
        OK (fluc_ttmlblend_frame_pool_acquire (ctx, FLUC_TTMLBLEND_FORMAT_NV12, W, H, 1, &f));
      }
      memset (f.plane[0], 0x55, (size_t) f.stride[0] * H);
      memset (f.plane[1], 0x80, (size_t) f.stride[1] * (H / 2));
    }
  }
  std::vector<uint64_t> tickets ((size_t) o.batch), prev_all;
  uint64_t prev = 0;
  double t_submit = 0, t_wait = 0;
  std::vector<uint64_t> ring;
  auto step = [&](int i) {
    if (const char *d = getenv ("E2E_DELAY_US"))
      usleep ((useconds_t) atoi (d));
    const double ta = now ();
    OK (fluc_ttmlblend_blend_host_many (ctx, (uint32_t) o.batch, streams.data (), FLUC_TTMLBLEND_FORMAT_NV12, W, H, 0,
            sets[i % n_sets].data (), tickets.data ()));
    t_submit += now () - ta;
    if (o.pageable) {           /* staged frames complete one by one: wait for each of the previous set */
      for (uint64_t t : prev_all)
        OK (fluc_ttmlblend_wait (ctx, t));
      prev_all = tickets;
      return;
    }
    const double tb = now ();
    ring.push_back (tickets.back ());
    if ((int) ring.size () > o.depth) {
      OK (fluc_ttmlblend_wait (ctx, ring.front ()));
      ring.erase (ring.begin ());
    }
    t_wait += now () - tb;
    (void) prev;
  };
  for (int i = 0; i < 4; i++)
    step (i);
  OK (fluc_ttmlblend_sync (ctx));
  fluc_ttmlblend_stats_reset (ctx);
  barrier (sh, G);
  const double t0 = now ();
  int n = 0;
  double t = 0;
  do {
    step (n++);
    step (n++);
    t = now () - t0;
  } while (t < o.secs);
  OK (fluc_ttmlblend_sync (ctx));
  t = now () - t0;
  FlucTtmlBlendStats st;
  fluc_ttmlblend_stats_copy (ctx, &st);
  if (getenv ("E2E_TIMES"))
    fprintf (stderr, "worker %d: %d steps, %.3f ms in blend_host_many and %.3f ms in wait per step\n", w, n + 4,
        t_submit / (n + 4) * 1e3, t_wait / (n + 4) * 1e3);
  sh->fps[w] = (double) n * o.batch / t;
  sh->gbs[w] = (double) st.h2d_bytes / t / 1e9;
  barrier (sh, G);
  fluc_ttmlblend_free (ctx);
}

int
main (int argc, char **argv)
{
  Options o;
  for (int i = 1; i < argc; i++) {
    const std::string a = argv[i];
    auto next = [&]() -> std::string { return i + 1 < argc ? argv[++i] : ""; };
    if (a == "--gpus") {
      const std::string s = next ();
      for (size_t b = 0; b <= s.size ();) {
        const size_t e = s.find (',', b);
        o.gpus.push_back (atoi (s.substr (b, e == std::string::npos ? std::string::npos : e - b).c_str ()));
        if (e == std::string::npos)
          break;
        b = e + 1;
      }
    } else if (a == "--threads")
      o.threads = true;
    else if (a == "--pin")
      o.pin = true;
    else if (a == "--opaque")
      o.opaque = true;
    else if (a == "--pageable")
      o.pageable = true;
    else if (a == "--secs")
      o.secs = atof (next ().c_str ());
    else if (a == "--batch")
      o.batch = atoi (next ().c_str ());
    else if (a == "--depth")
      o.depth = std::max (1, std::min (6, atoi (next ().c_str ())));
    else
      return 2;
  }
  if (o.gpus.empty ())
    o.gpus.push_back (0);
  const int G = (int) o.gpus.size ();
  if (G > kMaxGpus)
    return 2;
  Shared *sh = (Shared *) mmap (nullptr, sizeof (Shared), PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
  memset ((void *) sh, 0, sizeof *sh);
  if (o.threads) {
    std::vector<std::thread> th;
    for (int w = 0; w < G; w++)
      th.emplace_back (worker, std::cref (o), w, sh);
    for (auto &t : th)
      t.join ();
  } else {
    std::vector<pid_t> kids;
    for (int w = 0; w < G; w++) {
      const pid_t pid = fork ();
      if (pid == 0) {
        worker (o, w, sh);
        _exit (0);
      }
      kids.push_back (pid);
    }
    int bad = 0;
    for (pid_t k : kids) {
      int st = 0;
      waitpid (k, &st, 0);
      if (!WIFEXITED (st) || WEXITSTATUS (st) != 0) {
        bad++;
        sh->failed.store (1);
      }
    }
    if (bad)
      return 1;
  }
  double fps = 0, gbs = 0;
  for (int w = 0; w < G; w++) {
    fps += sh->fps[w];
    gbs += sh->gbs[w];
  }
  const char *sy = getenv ("FLUC_TTMLBLEND_SYNC");
  printf ("e2e %d GPU(s) as %s, pin=%d sync=%s %s: %9.0f frames/s aggregate, %6.1f GB/s each way; per GPU:",
      G, o.threads ? "threads" : "processes", o.pin ? 1 : 0, sy ? sy : "spin",
      o.pageable ? (o.opaque ? "opaque, pageable frames" : "translucent, pageable frames") : o.opaque ? "opaque" : "translucent", fps, gbs);
  for (int w = 0; w < G; w++)
    printf (" %.0f", sh->fps[w]);
  printf ("\n");
  return 0;
}
