"""What stream-ordered submission buys a CUDA pipeline: the frames of config 3 (4K NV12, two
full-width cue regions, 32 frames per step) handed over by a producer stream and read back by a
consumer stream, three ways, alternated over two rounds in one process:

  (a) stream-ordered  producer kernel -> submit_many_after -> wait_on_stream -> consumer kernel,
                      no host synchronisation inside the loop
  (b) host-ordered    producer kernel -> synchronize -> submit_many -> wait -> consumer kernel,
                      the only correct hand-over without (a)
  (c) blend alone     submit_many_repeat, bench.py's loop

The producer is one torch kernel that writes the first luma row of each of the step's 32 source
frames: it stands in for a decoder's completion, not for its bandwidth. The consumer is one torch
kernel that reads the first luma row of each destination frame (an encoder's start). (a) and (b)
rotate 4 sets of sources and 4 of destinations, as decoder and encoder pools do; the producer of a
step waits on the device for the consumer that last read its destination set, and (a) orders it
after the blend that last read its source set with wait_on_stream. (c) rotates 4 destination sets
over one source set, like bench.py. Every set of 32 frames is 398 MB, larger than the 126 MB L2.

  python tools/stream_order_probe.py [--steps 200] [--warmup 20]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

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
    wl, tb = pkg.workloads, pkg.ttmlblend
    cfg = wl.CONFIGS[3]
    W, H, n = cfg.width, cfg.height, cfg.batch
    ctx = pkg.TtmlBlend(0)
    ctx.overlay_set(1, wl.overlay_for(cfg), wl.region_rects(cfg))
    base = wl.frame_for(cfg, 0, "NV12")
    y_bytes = W * H
    fb = wl.frame_bytes("NV12", W, H)
    one = torch.from_numpy(np.concatenate([p.ravel() for p in base])).cuda()

    def frame_set():
        t = torch.empty((n, fb), dtype=torch.uint8, device="cuda")
        t.copy_(one.expand(n, fb))
        return t

    def frames(t):
        out = []
        for i in range(n):
            f = tb.Frame()
            f.plane[0], f.stride[0] = t[i].data_ptr(), W
            f.plane[1], f.stride[1] = t[i].data_ptr() + y_bytes, W
            out.append(f)
        return out

    srcs = [frame_set() for _ in range(SETS)]
    dsts = [frame_set() for _ in range(SETS)]
    batches = [ctx.Batch([1] * n, "NV12", W, H, frames(srcs[k]), frames(dsts[k])) for k in range(SETS)]
    bench_batch = ctx.Batch([1] * n, "NV12", W, H, frames(srcs[0]), [f for d in dsts for f in frames(d)])
    sink = torch.empty((n, W), dtype=torch.uint8, device="cuda")
    prod, cons = torch.cuda.Stream(), torch.cuda.Stream()
    read_done = [torch.cuda.Event() for _ in range(SETS)]   # the consumer has read destination set k
    src_ticket = [0] * SETS                                 # newest blend that read source set k
    torch.cuda.synchronize()

    def produce(step):
        k = step % SETS
        prod.wait_event(read_done[k])
        with torch.cuda.stream(prod):
            srcs[k][:, :W].fill_(step & 255)

    def consume(step):
        k = step % SETS
        with torch.cuda.stream(cons):
            sink.copy_(dsts[k][:, :W])
            read_done[k].record(cons)

    def stream_ordered(steps, first):
        for s in range(first, first + steps):
            k = s % SETS
            if src_ticket[k]:
                ctx.wait_on_stream(src_ticket[k], prod.cuda_stream)
            produce(s)
            t = ctx.submit_many_after(batches[k], prod.cuda_stream)[n - 1]
            src_ticket[k] = t
            ctx.wait_on_stream(t, cons.cuda_stream)
            consume(s)

    def host_ordered(steps, first):
        for s in range(first, first + steps):
            produce(s)
            prod.synchronize()
            t = ctx.submit_many(batches[s % SETS])[n - 1]
            ctx.wait(t)
            consume(s)

    def blend_alone(steps, first):
        ctx.submit_many_repeat(bench_batch, steps)

    loops = [("a", "stream-ordered: producer -> submit_many_after -> wait_on_stream -> consumer", stream_ordered),
             ("b", "host-ordered: producer -> synchronize -> submit_many -> wait -> consumer", host_ordered),
             ("c", "blend alone: submit_many_repeat (bench.py's loop)", blend_alone)]
    print(f"GPU 0: {gpu_identity()}")
    print(f"workload: config 3 ({W}x{H} NV12, {n} frames per step, two full-width cue regions), "
          f"{args.steps} timed steps after {args.warmup} warm-up steps per loop and round; "
          f"{n * fb / 1e6:.0f} MB per frame set")
    step = 0
    results = {}
    for rnd in range(2):
        for key, what, fn in loops:
            fn(args.warmup, step)
            step += args.warmup
            torch.cuda.synchronize()
            ctx.sync()
            ctx.stats_reset()
            t0 = time.perf_counter()
            fn(args.steps, step)
            step += args.steps
            torch.cuda.synchronize()
            ctx.sync()
            dt = time.perf_counter() - t0
            st = ctx.stats()
            fps = args.steps * n / dt
            results.setdefault(key, []).append(fps)
            print(f"round {rnd} ({key}) {what}: {fps / 1e3:8.1f} k frames/s, {dt / args.steps * 1e3:.4f} ms per step, "
                  f"{st['launches'] / args.steps:.2f} launches per step, "
                  f"{st['dependent_launches'] / args.steps:.2f} dependent launches per step")
    print("summary (k frames/s, round 0 / round 1): " +
          ", ".join(f"({k}) {r[0] / 1e3:.1f} / {r[1] / 1e3:.1f}" for k, r in results.items()))
    ctx.close()


if __name__ == "__main__":
    main()
