"""What a resize costs: config 3 (4K NV12, two cue regions, 32 frames per step) with the cue's
rectangles resized before every step, three ways, alternated over two rounds in one process:

  (a) fixed       the rectangles installed scaled, at the first of two render sizes, untouched
  (b) resize      overlay_set_render_rectangles before every step, alternating between the two
                  scaled render sizes (9/8 and 7/8 of the pixel size), then submit_many + flush
  (c) reinstall   overlay_set_rectangles of the same rectangles with the new render size before
                  every step: the only way to resize before overlay_set_render_rectangles

and the same three with one frame per step (the cue changes size for every frame). Each step
writes one of 4 destination sets of 32 frames (398 MB, larger than the 126 MB L2) from one
source set of 32 frames, like bench.py. Times are host clocks around whole loops that end in a
device sync.

Afterwards the resize call itself: a host clock around each overlay_set_render_rectangles call
(which returns once the scale-and-scan kernel and the readback of its row spans have finished,
and the prepare has been queued), and, in a separate pass under torch.profiler with CUDA
activities, the device time of the scale-and-scan kernel and of the copies around it: the part
of the call's host wait that is GPU work.

  python tools/resize_probe.py [--steps 200] [--warmup 20] [--out FILE]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402

SETS = 4


def gpu_identity():
    """Name and power limit of GPU 0, read in the same run as the numbers (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"unknown ({e})"
    return out or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--calls", type=int, default=200, help="resize calls timed one by one")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    pkg = graft.load_package()
    wl = pkg.workloads
    cfg = wl.CONFIGS[3]
    W, H, n = cfg.width, cfg.height, cfg.batch
    ctx = pkg.TtmlBlend(0)
    img = wl.overlay_for(cfg)
    boxes = wl.region_rects(cfg)
    sizes = [[(w * 9 // 8, h * 9 // 8) for _, _, w, h in boxes], [(w * 7 // 8, h * 7 // 8) for _, _, w, h in boxes]]

    def render(s):
        return [(x, y, rw, rh) for (x, y, _, _), (rw, rh) in zip(boxes, sizes[s % 2])]

    def rectangles(s):
        return [dict(pixels=img[y:y + h, x:x + w], x=x, y=y, premultiplied=True, render_width=rw, render_height=rh)
                for (x, y, w, h), (rw, rh) in zip(boxes, sizes[s % 2])]

    ctx.overlay_set_rectangles(1, rectangles(0))
    srcs = [ctx.acquire("NV12", W, H) for _ in range(n)]
    for i, s_ in enumerate(srcs):
        s_.upload(wl.frame_for(cfg, i, "NV12"))
    dsts = [[ctx.acquire("NV12", W, H) for _ in range(n)] for _ in range(SETS)]
    batches = [ctx.Batch([1] * n, "NV12", W, H, [s_.c for s_ in srcs], [d.c for d in dsts[k]]) for k in range(SETS)]
    singles = [ctx.Batch([1], "NV12", W, H, [srcs[i].c], [dsts[k][i].c]) for k in range(SETS) for i in range(n)]

    def run(batch_of, change):
        def loop(steps, first):
            for s in range(first, first + steps):
                change(s)
                ctx.submit_many(batch_of(s))
                ctx.flush()
        return loop

    fixed = lambda s: None                                                    # noqa: E731
    resize = lambda s: ctx.overlay_set_render_rectangles(1, render(s))        # noqa: E731
    reinstall = lambda s: ctx.overlay_set_rectangles(1, rectangles(s))        # noqa: E731
    step_batch = lambda s: batches[s % SETS]                                  # noqa: E731
    frame_batch = lambda s: singles[s % len(singles)]                         # noqa: E731
    loops = [("a", n, "fixed size", fixed),
             ("b", n, "resize: overlay_set_render_rectangles before every step", resize),
             ("c", n, "reinstall: overlay_set_rectangles at the new size before every step", reinstall),
             ("a1", 1, "fixed, one frame per step", fixed),
             ("b1", 1, "resize before every frame", resize),
             ("c1", 1, "reinstall before every frame", reinstall)]
    say(f"GPU 0: {gpu_identity()}")
    say(f"workload: config 3 ({W}x{H} NV12, {len(boxes)} cue regions {[(w, h) for _, _, w, h in boxes]} rendered "
        f"at {sizes[0]} / {sizes[1]}), {args.steps} timed steps after {args.warmup} warm-up steps per loop and "
        f"round; 32-frame steps rotate {SETS} destination sets")
    step = 0
    results = {}
    for rnd in range(2):
        for key, per_step, what, change in loops:
            fn = run(step_batch if per_step == n else frame_batch, change)
            ctx.overlay_set_rectangles(1, rectangles(step))
            fn(args.warmup, step)
            step += args.warmup
            ctx.sync()
            ctx.stats_reset()
            t0 = time.perf_counter()
            fn(args.steps, step)
            step += args.steps
            ctx.sync()
            dt = time.perf_counter() - t0
            st = ctx.stats()
            fps = args.steps * per_step / dt
            results.setdefault(key, []).append(fps)
            say(f"round {rnd} ({key}) {what}: {fps / 1e3:8.2f} k frames/s, {dt / args.steps * 1e3:.4f} ms per step, "
                f"{st['launches'] / args.steps:.2f} launches, {st['prepare_launches'] / args.steps:.2f} "
                f"prepare launches and {st['h2d_bytes'] / args.steps / 1e3:.1f} kB host-to-device per step")
    say("summary (k frames/s, round 0 / round 1): " +
        ", ".join(f"({k}) {r[0] / 1e3:.2f} / {r[1] / 1e3:.2f}" for k, r in results.items()))

    # the call alone: host clock around each call, the blend idle
    ctx.overlay_set_rectangles(1, rectangles(0))
    ctx.wait(ctx.submit_many(batches[0])[-1])
    ctx.sync()
    calls = []
    for s in range(1, args.calls + 1):
        t0 = time.perf_counter()
        ctx.overlay_set_render_rectangles(1, render(s))
        calls.append(time.perf_counter() - t0)
        ctx.sync()
    calls.sort()
    say(f"overlay_set_render_rectangles alone ({args.calls} calls, device idle before each): median "
        f"{calls[len(calls) // 2] * 1e6:.1f} us, p10 {calls[len(calls) // 10] * 1e6:.1f} us, "
        f"p90 {calls[9 * len(calls) // 10] * 1e6:.1f} us per call")
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for s in range(1, 51):
                ctx.overlay_set_render_rectangles(1, render(s))
                ctx.sync()
        kern, copies, nk, nc = 0.0, 0.0, 0, 0
        for e in prof.events():
            name = e.name
            dt = getattr(e, "device_time", None)
            if dt is None:
                dt = e.cuda_time
            if "scale_scan_batch" in name:
                kern += dt
                nk += 1
            elif "Memcpy" in name and ("DtoH" in name or "HtoD" in name):
                copies += dt
                nc += 1
        if nk:
            say(f"profiled (50 calls): ttmlblend_scale_scan_batch_kernel {kern / nk:.1f} us per call ({nk} launches), "
                f"host<->device copies {copies / 50:.1f} us per call ({nc} copies)")
        else:
            say("profiled: no scale-and-scan kernel in the trace (not measured)")
    except Exception as e:      # the numbers above stand without it
        say(f"profiled: not measured ({type(e).__name__}: {e})")
    for f in srcs + [d for s in dsts for d in s]:
        f.release()
    ctx.close()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
