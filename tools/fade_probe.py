"""What a fade costs: config 3 (4K NV12, two cue regions, 32 frames per step) with the cue's
global alpha changed before every step, three ways, alternated over two rounds in one process:

  (a) fixed       global alpha 1.0 all along, submit_many + flush per step
  (b) set_alpha   overlay_set_global_alpha with a new value before every step (every frame faded:
                  the values stay below 1), then the same submit_many + flush
  (c) reinstall   overlay_set_rectangles of the same rectangles (the cue's region boxes of
                  ttmlrender's image, premultiplied) with the new global_alpha before every step:
                  the only way to fade before overlay_set_global_alpha

and the same three with one frame per step (the value changes for every frame). Each step
writes one of 4 destination sets of 32 frames (398 MB, larger than the 126 MB L2) from one
source set of 32 frames, like bench.py. Times are host clocks around whole loops that end in a
device sync. Afterwards (a) and (b) run once more with every launch timed by an event pair on
the blend stream (set_profiling: launches then do not overlap), which splits a step into
kernel time and what lies between the kernels.

  python tools/fade_probe.py [--steps 200] [--warmup 20]
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
    args = ap.parse_args()
    pkg = graft.load_package()
    wl = pkg.workloads
    cfg = wl.CONFIGS[3]
    W, H, n = cfg.width, cfg.height, cfg.batch
    ctx = pkg.TtmlBlend(0)
    img = wl.overlay_for(cfg)
    boxes = wl.region_rects(cfg)

    def rectangles(alpha):
        return [dict(pixels=img[y:y + h, x:x + w], x=x, y=y, global_alpha=alpha, premultiplied=True)
                for x, y, w, h in boxes]

    ctx.overlay_set_rectangles(1, rectangles(1.0))
    srcs = [ctx.acquire("NV12", W, H) for _ in range(n)]
    for i, s_ in enumerate(srcs):
        s_.upload(wl.frame_for(cfg, i, "NV12"))
    dsts = [[ctx.acquire("NV12", W, H) for _ in range(n)] for _ in range(SETS)]
    batches = [ctx.Batch([1] * n, "NV12", W, H, [s_.c for s_ in srcs], [d.c for d in dsts[k]]) for k in range(SETS)]
    singles = [ctx.Batch([1], "NV12", W, H, [srcs[i].c], [dsts[k][i].c]) for k in range(SETS) for i in range(n)]

    def value(s):
        return 0.3 + 0.6 * ((s * 37) % 101) / 101        # below 1: every frame is faded

    def run(batch_of, change):
        def loop(steps, first):
            for s in range(first, first + steps):
                change(s)
                ctx.submit_many(batch_of(s))
                ctx.flush()
        return loop

    fixed = lambda s: None                               # noqa: E731
    set_alpha = lambda s: ctx.overlay_set_global_alpha(1, value(s))            # noqa: E731
    reinstall = lambda s: ctx.overlay_set_rectangles(1, rectangles(value(s)))   # noqa: E731
    step_batch = lambda s: batches[s % SETS]             # noqa: E731
    frame_batch = lambda s: singles[s % len(singles)]    # noqa: E731
    loops = [("a", n, "fixed: global alpha 1.0", fixed),
             ("b", n, "set_alpha: overlay_set_global_alpha before every step", set_alpha),
             ("c", n, "reinstall: overlay_set_rectangles with the new global_alpha before every step", reinstall),
             ("a1", 1, "fixed, one frame per step", fixed),
             ("b1", 1, "set_alpha before every frame", set_alpha),
             ("c1", 1, "reinstall before every frame", reinstall)]
    print(f"GPU 0: {gpu_identity()}")
    print(f"workload: config 3 ({W}x{H} NV12, {len(boxes)} cue regions), {args.steps} timed steps after "
          f"{args.warmup} warm-up steps per loop and round; 32-frame steps rotate {SETS} destination sets")
    step = 0
    results = {}
    for rnd in range(2):
        for key, per_step, what, change in loops:
            fn = run(step_batch if per_step == n else frame_batch, change)
            ctx.overlay_set_rectangles(1, rectangles(1.0))
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
            print(f"round {rnd} ({key}) {what}: {fps / 1e3:8.2f} k frames/s, {dt / args.steps * 1e3:.4f} ms per step, "
                  f"{st['launches'] / args.steps:.2f} launches and {st['prepare_launches'] / args.steps:.2f} "
                  f"prepare launches per step")
    print("summary (k frames/s, round 0 / round 1): " +
          ", ".join(f"({k}) {r[0] / 1e3:.2f} / {r[1] / 1e3:.2f}" for k, r in results.items()))
    for key, per_step, what, change in loops[:2]:
        fn = run(step_batch, change)
        ctx.overlay_set_rectangles(1, rectangles(1.0))
        fn(args.warmup, step)
        step += args.warmup
        ctx.sync()
        ctx.set_profiling(1)
        ctx.stats_reset()
        fn(args.steps // 4, step)
        step += args.steps // 4
        ctx.sync()
        st = ctx.stats()
        ctx.set_profiling(0)
        print(f"profiled ({key}): {st['kernel_ms'] / max(1, st['kernel_ms_launches']):.4f} ms of kernel per launch "
              f"over {st['kernel_ms_launches']} launches")
    for f in srcs + [d for s in dsts for d in s]:
        f.release()
    ctx.close()


if __name__ == "__main__":
    main()
