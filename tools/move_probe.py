"""What a move costs: config 3 (4K NV12, two cue regions, 32 frames per step) with the cue's
rectangles moved before every step, three ways, alternated over two rounds in one process:

  (a) fixed       the rectangles where they were installed, submit_many + flush per step
  (b) move        overlay_set_positions before every step, to a position whose x and y parity
                  both differ from the step before (a scroll), then the same submit_many + flush
  (c) reinstall   overlay_set_rectangles of the same rectangles at the new position before every
                  step: the only way to move a cue before overlay_set_positions

and the same three with one frame per step (the cue moves for every frame). Each step writes one
of 4 destination sets of 32 frames (398 MB, larger than the 126 MB L2) from one source set of 32
frames, like bench.py. Times are host clocks around whole loops that end in a device sync.

  python tools/move_probe.py [--steps 200] [--warmup 20] [--out FILE]
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

    def offset(s):
        """x and y parity flip at every step; the cue sweeps 32 columns and 4 rows and comes back."""
        return s % 32 - 16, s % 4 - 2

    def rectangles(s):
        dx, dy = offset(s)
        return [dict(pixels=img[y:y + h, x:x + w], x=x + dx, y=y + dy, premultiplied=True) for x, y, w, h in boxes]

    def positions(s):
        dx, dy = offset(s)
        return [x + dx for x, _, _, _ in boxes], [y + dy for _, y, _, _ in boxes]

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

    fixed = lambda s: None                                             # noqa: E731
    move = lambda s: ctx.overlay_set_positions(1, *positions(s))       # noqa: E731
    reinstall = lambda s: ctx.overlay_set_rectangles(1, rectangles(s))  # noqa: E731
    step_batch = lambda s: batches[s % SETS]                           # noqa: E731
    frame_batch = lambda s: singles[s % len(singles)]                  # noqa: E731
    loops = [("a", n, "fixed position", fixed),
             ("b", n, "move: overlay_set_positions before every step", move),
             ("c", n, "reinstall: overlay_set_rectangles at the new position before every step", reinstall),
             ("a1", 1, "fixed, one frame per step", fixed),
             ("b1", 1, "move before every frame", move),
             ("c1", 1, "reinstall before every frame", reinstall)]
    say(f"GPU 0: {gpu_identity()}")
    say(f"workload: config 3 ({W}x{H} NV12, {len(boxes)} cue regions), {args.steps} timed steps after "
        f"{args.warmup} warm-up steps per loop and round; 32-frame steps rotate {SETS} destination sets")
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
    for f in srcs + [d for s in dsts for d in s]:
        f.release()
    ctx.close()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
