#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: frames/s and % of the HBM roofline for the 4K NV12
TTML overlay blend (config 3: 3840x2160 NV12, two full-width cue regions, 32 frames per
launch), with the reference's CPU blend timed beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 3]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one launch of the blend over one batch (32 device-resident 4K frames,
src -> dst, whole frame read and written; 398 MB in + 398 MB out per step, i.e. inputs
larger than the 126 MB L2). Per-GPU work is fixed as N grows (weak scaling, each rank its
own frame batches, no collective on the data path); torch.distributed is only used for the
barrier, the MAX over ranks of the device time and a gather of the result records.

Numbers in the JSON line (every figure of `roofline` can be recomputed from the line itself
plus profiles/r02_roofline_traffic.json):
  value         frames/s, frames resident in HBM, CUDA-event time on the blend stream, K steps.
  roofline      achieved = algorithmic bytes per launch (BASELINE.md: frame read + frame write +
                4 B/px overlay) / launch_ms, launch_ms = device time of the timed region / its
                launches (back-to-back launches of the one kernel; an event pair around every
                n-th launch is the cross-check, `launch_ms_event_pairs`); frac against
                MEASURED_PEAKS.json; traffic = ncu dram bytes per launch FOR THIS WORKLOAD
                (profiles/r02_roofline_traffic.json) and frac_dram = traffic / launch_ms / peak.
  sustained     the same steps repeated for ~1.5 s: frames/s and the nvidia-smi clocks of that
                very window (the timed region of 20 steps lasts 2.4 ms, too short to sample).
  distinct_cues 32 frames of 32 streams with 32 different 4K cues: 186 MB of prepared overlay,
                more than L2, so the overlay really streams from HBM (config 3 only).
  e2e           frames/s through fluc_ttmlblend_blend_host_many (the drop-in for
                gst_video_overlay_composition_blend): pinned HOST frames, the rows the overlay
                touches cross PCIe both ways inside the timed region (`transport`: zero copy or
                the copy engines, whichever the library's own timed trial found faster on this
                GPU); pcie_ceiling_gbs is what the same traffic reaches with no blend in it -- a
                kernel rewriting host memory in place, or the copy engine both ways, the larger
                -- measured in the same run on all ranks at once, frac_of_pcie = e2e bytes/s per
                direction over it. `pageable`:
                the same through ordinary (not pinned) host memory.
  cfg5          BASELINE config 5 beside the headline: 256 1080p I420 streams sharded
                stream % N over the ranks (strong scaling).
  multi         (N > 1) rank 0 alone drives all N GPUs from one process through
                FlucTtmlBlendMulti while the other ranks idle.
  cpu_baseline  the CPU oracle (a port of gst_video_blend: GStreamer is not installable here)
                on this box's host cores, bounded sample, rank 0 at N=1 only.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import __graft_entry__ as graft  # noqa: E402

DST_SETS = 4
METRIC = "frames/sec, 4K NV12 TTML overlay blend"
UNIT = "frames/s"
DUMP_BYTES = 60 << 20       # --dump-outputs: the .npy files stay below 64 MB in all


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:   # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(workload: str, fmt: str):
    """ncu dram__bytes_read.sum + dram__bytes_write.sum per launch for this workload, or None."""
    p = os.path.join(ROOT, "profiles", "r02_roofline_traffic.json")
    try:
        table = json.load(open(p))
    except Exception:   # noqa: BLE001
        return None, None
    rec = table.get(f"{workload}:{fmt}") or table.get(workload)
    if not rec:
        return None, None
    # per frame: a rank of a sharded run launches fewer frames than the capture did
    return rec.get("dram_bytes_per_frame"), rec.get("source")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under load."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0: float, t1: float):
        rows = [s for t, s in self.samples if t0 <= t <= t1]
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                smax = max(smax, float(f[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus: int):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    device = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's version / debug lines go to stdout by default: keep stdout for the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            device = torch.device("cuda", local)
            dist_mod.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
        else:
            dist_mod.init_process_group("gloo", rank=rank, world_size=world)
        dist = dist_mod
    return dist, device, world, rank, local


def cpu_barrier(dist, group):
    """A barrier that does not occupy the GPUs (an NCCL barrier is a kernel that spins until every
    rank has arrived): used while rank 0 alone drives all devices."""
    if dist is not None:
        dist.barrier(group=group)


def barrier(dist, device):
    if dist is not None:
        if device is not None:
            import torch
            torch.cuda.synchronize(device)
        dist.barrier()


def config_record(cfg, wl, fmt, world):
    """The `config` object: the same keys and values in both arms (this one and --impl reference)."""
    W, H = cfg.width, cfg.height
    batch = cfg.batch if cfg.streams == 1 else cfg.streams
    per_step_bytes = batch * wl.frame_bytes(fmt, W, H)
    return {"workload": cfg.name, "format": fmt, "width": W, "height": H,
            "frames_per_step": batch,
            "streams": cfg.streams, "regions": [list(r) for r in wl.region_rects(cfg)],
            "overlay": "ttmlrender's frame-sized premultiplied BGRA image (W*H*4, cleared, regions drawn in)",
            "mode": "out-of-place (whole frame read + written)",
            "buffers": f"one set of source frames, results rotate through {DST_SETS} sets of destination frames",
            "bytes_per_frame": wl.algorithmic_bytes(cfg, fmt),
            "l2": (f"inputs larger than L2 ({per_step_bytes / 1e6:.0f} MB read + as much written per step, "
                   "L2 is 126 MB)" if per_step_bytes > 126e6 else
                   "inputs fit in L2 (small config); no flush between steps"),
            "parallelism": (f"{cfg.streams} streams sharded stream % N, no collective" if cfg.streams > 1
                            else "N x independent frame batches, no collective")}


# ---------------------------------------------------------------------------
# CPU legs (the only places bench.py touches oracle/)

def cpu_frames(cfg, wl, n_frames):
    """n_frames fresh source frames, the same as the GPU arm's (frame i rolled by 16 i pixels)."""
    from oracle import oracle
    base = wl.frame_for(cfg, 0)
    keep = []
    arr = (oracle.RefFrame * n_frames)()
    for i in range(n_frames):
        planes = [np.roll(p, i * 16, axis=1).copy() for p in base]
        keep.append(planes)
        arr[i] = oracle.make_frame(cfg.fmt, cfg.width, cfg.height, planes)
    return arr, keep


def cpu_reference_setup(cfg, wl, n_frames):
    from oracle import oracle
    lib = oracle.load(native=True, out_dir=tempfile.mkdtemp(prefix="ttmlblend_oracle_"))
    ov = wl.overlay_for(cfg)
    arr, keep = cpu_frames(cfg, wl, n_frames)
    rects = oracle.make_rectangles(oracle.ttmlrender_rectangles(ov))
    return lib, arr, rects, keep, ov


def cpu_blend_fps(lib, arr, rects, n_frames, threads):
    secs = lib.tbref_blend_many(arr, n_frames, rects, 1, threads)
    return n_frames / secs, secs


def run_cpu_baseline(cfg, wl, target_s=12.0):
    cores = os.cpu_count() or 1
    probe_n = max(cfg.batch, min(cfg.streams, 32), os.cpu_count() or 1)
    lib, arr, rects, keep, ov = cpu_reference_setup(cfg, wl, probe_n)
    fps, secs = cpu_blend_fps(lib, arr, rects, probe_n, cores)       # probe (also warms caches)
    rounds = max(1, int(target_s / max(secs, 1e-3)))
    t = 0.0
    for _ in range(rounds):
        _, s = cpu_blend_fps(lib, arr, rects, probe_n, cores)
        t += s
    n = rounds * probe_n
    # for transparency: the same CPU code if someone cropped the image to the region boxes first
    # (the reference does not: ttmlrender pushes the whole frame-sized image downstream)
    from oracle import oracle
    crop = [dict(pixels=ov[r.y:r.y + r.h, r.x:r.x + r.w], x=r.x, y=r.y) for r in cfg.regions]
    crop_rects = oracle.make_rectangles(crop)
    t_crop = lib.tbref_blend_many(arr, probe_n, crop_rects, len(crop), cores)
    t_crop = min(t_crop, lib.tbref_blend_many(arr, probe_n, crop_rects, len(crop), cores))
    return {"value": n / t, "unit": UNIT, "cores": cores, "kind": "port",
            "value_if_cropped_to_regions": probe_n / t_crop,
            "sample": f"{n} frames of {cfg.width}x{cfg.height} {cfg.fmt} ({probe_n} buffers re-blended "
                      f"{rounds}x), ttmlrender's frame-sized premultiplied BGRA image as one "
                      f"rectangle (what the reference pipeline blends), oracle/ttmlblend_ref.c "
                      f"-O3 -march=native, {cores} pthreads, {t:.1f} s"}


def dump_rows(wl, shapes, n_frames):
    """Row numbers kept per plane by --dump-outputs: every row when the float32 copy of all
    frames fits DUMP_BYTES, else the same seeded sample of rows in every frame."""
    total = 4 * n_frames * sum(r * c for r, c in shapes)
    frac = min(1.0, DUMP_BYTES / total)
    rows = []
    for i, (r, _) in enumerate(shapes):
        k = max(1, int(r * frac))
        rows.append(np.sort(np.argsort(wl.splitmix64(0x64756D70 + i, r), kind="stable")[:k]))
    return rows


def dump_outputs(out_dir, frames, rows):
    """frames: per frame, the `rows` (dump_rows) of its planes as the caller receives them.
    Writes plane<i>.npy, float32 [frame, row, byte], and plane<i>_rows.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    for i, keep in enumerate(rows):
        np.save(os.path.join(out_dir, f"plane{i}.npy"), np.stack([f[i] for f in frames]).astype(np.float32))
        np.save(os.path.join(out_dir, f"plane{i}_rows.npy"), keep.astype(np.float64))


def run_reference_arm(args, cfg, wl, world, rank, real_stdout):
    """--impl reference: the reference's CPU implementation of the path (oracle port; GStreamer
    cannot be installed here) on all host threads, 32 frames per step like the GPU arm. Rank 0 only."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = max(cfg.batch, cfg.streams)          # the GPU arm's frames per step
    lib, arr, rects, keep, ov = cpu_reference_setup(cfg, wl, per_step)
    for _ in range(args.warmup):
        cpu_blend_fps(lib, arr, rects, per_step, cores)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_blend_fps(lib, arr, rects, per_step, cores)[1]
    fps = per_step * args.steps / t
    if args.dump_outputs:
        # the timed frames have been blended in place warmup + steps times; one blend of fresh
        # frames is what a caller of one step receives (and what the GPU arm dumps)
        arr, keep = cpu_frames(cfg, wl, per_step)
        lib.tbref_blend_many(arr, per_step, rects, 1, cores)
        rows = dump_rows(wl, [p.shape for p in keep[0]], len(keep))
        dump_outputs(args.dump_outputs, [[p[k] for p, k in zip(f, rows)] for f in keep], rows)
    line = {
        "impl": "reference", "metric": METRIC if args.config == 3 else f"frames/sec, TTML overlay blend ({cfg.name})",
        "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak" if cfg.streams == 1 else "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_record(cfg, wl, args.format or cfg.fmt, world),
        "reference_note": "CPU port of gst_video_overlay_composition_blend (oracle/ttmlblend_ref.c, scalar C, "
                          "-O3 -march=native, one pthread per host core); GStreamer itself is not installed in "
                          "this image, so kind is \"port\"",
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{per_step} frames per step x {args.steps} steps, frame-sized overlay rectangle"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=real_stdout, flush=True)


# ---------------------------------------------------------------------------

def protect_stdout():
    """stdout carries exactly one JSON line. Native libraries (NCCL prints its version there) write
    to file descriptor 1 behind Python's back, so fd 1 is pointed at stderr for the whole run and
    the line goes to a private duplicate of the real stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


class DeviceWorkload:
    """Device-resident frames of one configuration on one context, ready to be stepped."""

    def __init__(self, ctx, wl, sh, cfg, fmt, world, rank, distinct_cues=False, stream_base=0):
        self.ctx, self.cfg, self.fmt = ctx, cfg, fmt
        W, H = cfg.width, cfg.height
        self.B = wl.algorithmic_bytes(cfg, fmt)
        if cfg.streams > 1:
            # config 5: independent streams, one frame each per step, sharded stream % world
            ids = [stream_base + s for s in sh.shard_streams(cfg.streams, world, rank)]
            ovs = [wl.overlay_for(cfg, stream=k) for k in range(4)]      # 4 distinct cue images, reused
            for s_id in ids:
                ctx.overlay_set(s_id, ovs[s_id % len(ovs)], wl.region_rects(cfg))
            self.scaling = "strong"
        elif distinct_cues:
            # one stream per frame, every stream with its own cue image (the same layout, other
            # pixels): nothing of the prepared overlay is shared between the frames of a launch
            ids = [stream_base + 1 + i for i in range(cfg.batch)]
            ov = wl.overlay_for(cfg)
            for i, s_id in enumerate(ids):
                ctx.overlay_set(s_id, np.ascontiguousarray(np.roll(ov, 16 * i, axis=1)), wl.region_rects(cfg))
            self.scaling = "weak"
        else:
            ids = [stream_base + 1] * cfg.batch
            self.overlay = wl.overlay_for(cfg)
            ctx.overlay_set(stream_base + 1, self.overlay, wl.region_rects(cfg))
            self.scaling = "weak"
        self.stream_ids = ids
        self.batch = len(ids)
        self.base = wl.frame_for(cfg, rank, fmt)
        self.srcs = [ctx.acquire(fmt, W, H) for _ in range(self.batch)]
        # the results rotate through DST_SETS sets of frames, as the frames of a running pipeline
        # come out of a buffer pool: a step does not land in the buffers of the step before it
        self.dst_sets = DST_SETS
        self.dsts = [ctx.acquire(fmt, W, H) for _ in range(self.batch * self.dst_sets)]
        for i, s in enumerate(self.srcs):
            s.upload([np.roll(p, i * 16, axis=1) for p in self.base])
        self.tb = ctx.Batch(ids, fmt, W, H, [s.c for s in self.srcs], [d.c for d in self.dsts])
        self.tb_inplace = ctx.Batch(ids, fmt, W, H, [s.c for s in self.srcs], [s.c for s in self.srcs])

    # submit_many_repeat keeps ONE step counter per context across calls and workloads: step k of
    # the context writes destination set k % dst_sets. Every call here goes through steps(),
    # which keeps the same count per context.
    repeats = {}

    def steps(self, n, inplace=False):
        """n steps, each one submit_many of the whole batch + flush, issued by a native loop."""
        self.ctx.submit_many_repeat(self.tb_inplace if inplace else self.tb, n)
        DeviceWorkload.repeats[self.ctx] = DeviceWorkload.repeats.get(self.ctx, 0) + n

    def last_outputs(self, rows):
        """The destination frames of the context's latest step, `rows` of each plane kept; that
        step must be one of this workload's out-of-place steps."""
        ofs = (DeviceWorkload.repeats[self.ctx] - 1) % self.dst_sets * self.batch
        return [[p[keep] for p, keep in zip(d.download(), rows)] for d in self.dsts[ofs:ofs + self.batch]]

    def release(self, keep_srcs=False):
        for f in self.dsts + ([] if keep_srcs else self.srcs):
            f.release()


def timed_region(ctx, work, steps, dist, device, pairs, inplace=False, after=None):
    """K steps between barriers: (device ms, stats of the region). Afterwards, outside the timed
    region, `after()` if given (while the frames still hold the last step's results), then
    `pairs` more launches each between its own CUDA-event pair: the duration of one
    launch running alone (a timed launch neither overlaps its predecessor's tail nor lets its
    successor overlap its own), the cross-check of the region's mean."""
    ctx.sync()
    ctx.stats_reset()
    barrier(dist, device)
    ctx.timer_begin()
    work.steps(steps, inplace)
    ms = ctx.timer_end()
    ctx.sync()
    barrier(dist, device)
    st = ctx.stats()
    if after is not None:
        after()
    if pairs:
        ctx.stats_reset()
        ctx.set_profiling(1)
        work.steps(pairs, inplace)
        ctx.sync()
        sp = ctx.stats()
        ctx.set_profiling(0)
        st["kernel_ms"], st["kernel_ms_launches"] = sp["kernel_ms"], sp["kernel_ms_launches"]
    return ms, st


def roofline_record(work, ms, st, steps, peak, peak_src, cfg_name, fmt, kernel):
    launches = max(1, int(st["launches"]))
    launch_ms = ms / launches
    bytes_per_launch = work.B * work.batch * steps / launches
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9 if launch_ms > 0 else 0.0
    pairs = int(st["kernel_ms_launches"])
    traffic, traffic_src = load_traffic(cfg_name, fmt)
    if traffic:
        traffic *= work.batch * steps / launches      # the table holds DRAM bytes per frame
    rec = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "traffic": traffic, "kernel": kernel, "launch_ms": launch_ms, "launches_timed": launches,
           "timing": "device time of the whole timed region (CUDA events on the blend stream) / its launches; "
                     "the region holds nothing but back-to-back launches of this kernel",
           "launch_ms_event_pairs": (st["kernel_ms"] / pairs) if pairs else None,
           "event_pairs": pairs,
           "event_pairs_note": "launches timed one by one right after the timed region: each waits for its "
                               "predecessor and is not overlapped by its successor, which the launches of the "
                               "timed region are (programmatic dependent launch)",
           "dependent_launches": int(st.get("dependent_launches", 0)),
           "algorithmic_bytes_per_launch": bytes_per_launch, "peak_source": peak_src,
           "frac_of_8000_nominal": achieved / 8000.0}
    if traffic and launch_ms > 0:
        # the same launch time against the bytes DRAM really moved (ncu, this workload): below the
        # algorithmic figure where the prepared overlay (3 B/px) is shared by the frames of a
        # launch and served from L2
        rec["traffic_gbs"] = traffic / (launch_ms * 1e-3) / 1e9
        rec["frac_dram"] = rec["traffic_gbs"] / peak
        rec["traffic_over_algorithmic"] = traffic / bytes_per_launch
        rec["traffic_source"] = traffic_src
    return rec


def kernel_name(fmt, launches_kind="group"):
    kind = "PLANE8" if fmt in ("I420", "NV12", "YV12", "NV21") else "PACKED"
    return f"ttmlblend_{launches_kind}_kernel<{kind}>"


def e2e_loop(ctx, batches, n_steps):
    """blend_host_many on alternating sets of host frames; waits for the set submitted one step
    earlier, so that a batch is handed over while the previous one is on the bus."""
    prev = None
    for i in range(n_steps):
        tickets = ctx.blend_host_many(batches[i & 1])   # one C call per batch of host frames
        if prev is not None:
            ctx.wait(prev)
        prev = tickets[len(tickets) - 1]                # tickets complete in order
    ctx.wait(prev)


def main():
    real_stdout = protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--format", default=None, help="override the config's frame format (config 4: RGBA/BGRA/AYUV)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the legs beside the headline (distinct cues, config 5, multi, pageable, in place)")
    ap.add_argument("--distinct-cues", action="store_true",
                    help="headline workload = the distinct-cues variant (one stream and cue image per frame): "
                         "for profiling that leg on its own")
    ap.add_argument("--opaque-boxes", action="store_true",
                    help="the config's regions with opacity 1.0 (probe: no frame read under opaque vectors)")
    ap.add_argument("--event-pairs", type=int, default=12,
                    help="launches timed one by one with a CUDA-event pair AFTER the timed region "
                         "(cross-check of launch_ms)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frames of the last step (rank 0's) to DIR as "
                         "plane<i>.npy, float32 [frame, row, byte], with the row numbers kept in "
                         "plane<i>_rows.npy: all rows, or the same seeded sample of rows in every frame "
                         "when the frames would exceed 60 MB as float32")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs --steps >= 1")
    args.warmup = max(args.warmup, 3)
    profile_every = args.event_pairs

    pkg = graft.load_package()
    wl = pkg.workloads
    sh = pkg.sharding
    cfg = wl.CONFIGS[args.config]
    if args.opaque_boxes:
        cfg = dataclasses.replace(cfg, name=cfg.name + "+opaque_boxes",
                                  regions=[dataclasses.replace(r, opacity=1.0) for r in cfg.regions])
    dist, device, world, rank, local = dist_setup(args.gpus)

    if args.impl == "reference":
        run_reference_arm(args, cfg, wl, world, rank, real_stdout)
        if dist is not None:
            dist.destroy_process_group()
        return

    ctx = pkg.TtmlBlend(local)             # raises without a GPU: there is no CPU fallback
    fmt, W, H = (args.format or cfg.fmt), cfg.width, cfg.height
    peak, peak_src = load_peaks()
    sampler = ClockSampler(local)
    extras = not args.no_extras

    # ---- headline: device-resident frames --------------------------------------------------
    work = DeviceWorkload(ctx, wl, sh, cfg, fmt, world, rank, distinct_cues=args.distinct_cues)
    batch = work.batch
    ctx.set_batch(min(batch, 1024), 0)     # one launch per `batch` frames, no linger timer
    work.steps(args.warmup)
    # small configs: W steps last microseconds; keep stepping (untimed) until the GPU has been busy
    # for 30 ms, so that the timed region does not start on idle clocks
    t_w = time.time()
    warm_extra = 0
    while time.time() - t_w < 0.03:
        work.steps(max(1, args.warmup))
        ctx.sync()
        warm_extra += max(1, args.warmup)
    dump = None
    if args.dump_outputs and rank == 0:
        def dump():
            rows = dump_rows(wl, [(r, rb) for rb, r in pkg.ttmlblend.plane_layout(fmt, W, H)], batch)
            dump_outputs(args.dump_outputs, work.last_outputs(rows), rows)
    ms, st = timed_region(ctx, work, args.steps, dist, device, profile_every, after=dump)
    worst_ms = sh.reduce_max(ms, dist, device)
    records = sh.gather_records((batch * args.steps, ms, st["kernel_ms"], st["kernel_ms_launches"]), dist, device)
    value = sh.aggregate_fps(records)
    roofline = roofline_record(work, ms, st, args.steps, peak, peak_src, cfg.name, fmt, kernel_name(fmt))
    gpu_launches = int(st["launches"])

    # ---- sustained: the same steps for ~1.5 s, clocks sampled in that very window -----------
    chunk = max(1, int(0.05 / max(ms / args.steps * 1e-3, 1e-6)))     # ~50 ms of steps per call
    ctx.sync()
    t_s0 = time.time()
    ctx.timer_begin()
    n_sus = 0
    while time.time() - t_s0 < 1.5:
        work.steps(chunk)
        n_sus += chunk
        ctx.sync()
    ms_sus = ctx.timer_end()
    t_s1 = time.time()
    clocks = sampler.summary(t_s0, t_s1)
    clocks["window"] = "the `sustained` leg: the timed region's own steps repeated for 1.5 s right after it"
    sustained = {"value": batch * n_sus / (ms_sus * 1e-3), "unit": UNIT, "steps": n_sus,
                 "ms_per_step": ms_sus / n_sus, "seconds": ms_sus * 1e-3,
                 "achieved_gbs": work.B * batch * n_sus / (ms_sus * 1e-3) / 1e9,
                 "frac": work.B * batch * n_sus / (ms_sus * 1e-3) / 1e9 / peak,
                 "clocks": {k: clocks[k] for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples")},
                 "note": "this rank; includes a host synchronisation every ~50 ms"}
    if roofline.get("traffic"):
        sustained["frac_dram"] = roofline["traffic"] * n_sus / (ms_sus * 1e-3) / 1e9 / peak

    # ---- in place (SURVEY 8d: B_inplace reported separately) -------------------------------
    inplace = None
    if extras:
        ms_ip, st_ip = timed_region(ctx, work, args.steps, dist, device, 0, inplace=True)
        inplace = {"value": batch * args.steps / (ms_ip * 1e-3), "unit": UNIT,
                   "bytes_per_frame": st_ip["algorithmic_bytes"] // max(1, st_ip["frames_blended"]),
                   "algorithmic_gbs": st_ip["algorithmic_bytes"] / (ms_ip * 1e-3) / 1e9,
                   "note": "dst == src: only the rows under the cue regions are read and written "
                           "(B_inplace = 2 x touched frame bytes + 4 B/px overlay); this rank only"}

    # ---- distinct cues: the prepared overlay exceeds L2 -------------------------------------
    distinct = None
    if extras and cfg.streams == 1 and cfg.batch > 1 and not args.distinct_cues:
        try:
            dw = DeviceWorkload(ctx, wl, sh, cfg, fmt, world, rank, distinct_cues=True, stream_base=1000)
            dw.steps(args.warmup)
            ms_d, st_d = timed_region(ctx, dw, args.steps, dist, device, profile_every)
            rec_d = sh.gather_records((dw.batch * args.steps, ms_d), dist, device)
            rl = roofline_record(dw, ms_d, st_d, args.steps, peak, peak_src, cfg.name + "+distinct_cues", fmt,
                                 kernel_name(fmt))
            distinct = {"value": sh.aggregate_fps(rec_d), "unit": UNIT, "ms_per_step": ms_d / args.steps,
                        "launches": int(st_d["launches"]), "multi_launches": int(st_d["multi_launches"]),
                        "prepared_overlay_bytes": int(st_d["cache_bytes"]),
                        "roofline": rl,
                        "note": f"{dw.batch} frames per launch from {dw.batch} streams, each stream with its own "
                                "4K cue image: no overlay byte is shared between the frames of a launch"}
            dw.release()
            for s_id in dw.stream_ids:
                ctx.overlay_clear(s_id)
        except Exception as e:      # noqa: BLE001
            distinct = {"failed": repr(e)}

    # ---- e2e: pinned host frames through the drop-in call, PCIe inside the timed region -----
    e2e = None
    if not args.no_e2e:
        work.release(keep_srcs=True)
        stream_ids = work.stream_ids
        base = work.base
        # two sets of host frames: a set is handed over while the previous one is still crossing
        # PCIe, as the buffers of a running pipeline are (one set would serialise host and bus)
        host_sets = [[ctx.acquire(fmt, W, H, on_host=True) for _ in range(batch)] for _ in range(2)]
        for hs in host_sets:
            for i, hf in enumerate(hs):
                for dstp, srcp in zip(hf.host_planes(), base):
                    dstp[...] = np.roll(srcp, i * 16, axis=1)
        e2e_steps = max(4, min(args.steps, 100))
        host_batches = [ctx.Batch(stream_ids, fmt, W, H, [hf.c for hf in hs], [hf.c for hf in hs])
                        for hs in host_sets]
        # warm-up: long enough for the library to have tried both ways of crossing PCIe (128 frames
        # each, fluc_ttmlblend_set_host_dma mode 2) and to have settled on the faster one
        e2e_loop(ctx, host_batches, max(args.warmup, 16))
        ctx.sync()
        ctx.stats_reset()
        barrier(dist, device)
        t0 = time.perf_counter()
        e2e_loop(ctx, host_batches, e2e_steps)
        ctx.sync()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        barrier(dist, device)
        st2 = ctx.stats()
        rec2 = sh.gather_records((batch * e2e_steps, e2e_ms, st2["h2d_bytes"], st2["d2h_bytes"]), dist, device)
        e2e_value = sh.aggregate_fps(rec2)
        # the ceiling of this traffic shape on this box right now: every rank at the same time moves
        # what one step moves, (1) with a kernel that rewrites pinned host memory in place and
        # nothing else (the zero-copy path without the blend), (2) with the copy engine both ways
        step_bytes = max(1 << 20, int(st2["h2d_bytes"] // e2e_steps))
        barrier(dist, device)
        zc = ctx.pcie_probe(1, step_bytes, 0.4)
        barrier(dist, device)
        dma = ctx.pcie_probe(0, step_bytes, 0.4)
        barrier(dist, device)
        ceil = sh.gather_records((zc, dma), dist, device)
        zc_total, dma_total = sum(r[0] for r in ceil), sum(r[1] for r in ceil)
        e2e_gbs = sum(r[2] for r in rec2) / (max(r[1] for r in rec2) * 1e-3) / 1e9
        e2e = {"value": e2e_value, "unit": UNIT,
               "h2d_bytes_per_step": st2["h2d_bytes"] // e2e_steps,
               "d2h_bytes_per_step": st2["d2h_bytes"] // e2e_steps,
               "steps": e2e_steps, "launches": st2["launches"], "host_frames_numa_node": ctx.numa_node(),
               "host_dma_batches": int(st2["host_dma_batches"]),
               "transport": "copy engines" if st2["host_dma_batches"] * 2 > st2["launches"] else "zero copy",
               "gbs_per_direction": e2e_gbs,
               "pcie_ceiling_gbs": max(zc_total, dma_total),
               "frac_of_pcie": e2e_gbs / max(zc_total, dma_total) if max(zc_total, dma_total) else None,
               "pcie_zero_copy_gbs": zc_total, "pcie_dma_both_gbs": dma_total,
               "pcie_ceiling_per_rank": [round(max(r[0], r[1]), 1) for r in ceil],
               "pcie_note": "measured in this run, all ranks at once, per direction, summed over ranks. "
                            "pcie_zero_copy_gbs: a kernel that reads and rewrites as many pinned host bytes per "
                            "iteration as one e2e step moves, nothing else (fluc_ttmlblend_pcie_probe mode 1); "
                            "pcie_dma_both_gbs: the copy engine both ways, one piece per direction (mode 0); "
                            "pcie_ceiling_gbs: the larger of the two. profiles/r02_pcie_ceiling_summary.md: beyond "
                            "one GPU the box's root complex, not the path, is the limit",
               "api": "fluc_ttmlblend_blend_host_many on pinned host frames, in place; two sets of host frames "
                      "alternate so that a batch is submitted while the previous one is on the bus. The library "
                      "measures which transport is faster on this GPU (`transport`): zero copy -- the kernel reads "
                      "the rows under the cue regions from host memory and writes them back over PCIe, one launch "
                      "per batch -- or the copy engines -- 2-D copies of those rows for 8 frames at a time into "
                      "device staging, blend there, copy back, three streams"}
        if extras and cfg.streams == 1:
            # the same layout with OPAQUE region boxes (opacity 1.0, the common broadcast style): the
            # result under an opaque vector does not depend on the frame, so in place the frame is
            # written without being read and crosses PCIe in one direction only. Beside the headline,
            # not instead of it (the headline cue is translucent: both directions).
            try:
                ocfg = dataclasses.replace(cfg, regions=[dataclasses.replace(r, opacity=1.0) for r in cfg.regions])
                ctx.overlay_set(2, wl.overlay_for(ocfg), wl.region_rects(ocfg))
                ob = [ctx.Batch([2] * batch, fmt, W, H, [hf.c for hf in hs], [hf.c for hf in hs]) for hs in host_sets]
                e2e_loop(ctx, ob, 4)
                ctx.sync()
                n_op = max(4, min(e2e_steps, 40))
                t0 = time.perf_counter()
                e2e_loop(ctx, ob, n_op)
                ctx.sync()
                e2e["same_layout_with_opaque_boxes"] = batch * n_op / (time.perf_counter() - t0)
            except Exception as e:      # noqa: BLE001
                e2e["same_layout_with_opaque_boxes"] = f"failed: {e!r}"
            # a caller that keeps THREE sets of host frames going (waits two batches behind), with the
            # default zero-copy path and with the opt-in host DMA batches (fluc_ttmlblend_set_host_dma:
            # copy engines both ways + blend in device staging). One GPU only: on GPUs that share a
            # host bridge both are bound by it (profiles/r02_pcie_ceiling_summary.md).
            if world == 1:
                try:
                    third = [ctx.acquire(fmt, W, H, on_host=True) for _ in range(batch)]
                    for i, hf in enumerate(third):
                        for dstp, srcp in zip(hf.host_planes(), base):
                            dstp[...] = np.roll(srcp, i * 16, axis=1)
                    host_sets.append(third)
                    hb3 = host_batches + [ctx.Batch(stream_ids, fmt, W, H, [hf.c for hf in third], [hf.c for hf in third])]

                    def deep_loop(n_steps):
                        ring = []
                        for i in range(n_steps):
                            t = ctx.blend_host_many(hb3[i % 3])
                            ring.append(t[len(t) - 1])
                            if len(ring) > 2:
                                ctx.wait(ring.pop(0))
                        for r in ring:
                            ctx.wait(r)

                    deep = {}
                    n_deep = max(6, min(e2e_steps, 60))
                    for name, on in (("zero_copy", False), ("host_dma", True)):
                        ctx.set_host_dma(1 if on else 0)
                        deep_loop(6)
                        ctx.sync()
                        before = ctx.stats()["host_dma_batches"]
                        t0 = time.perf_counter()
                        deep_loop(n_deep)
                        ctx.sync()
                        deep[name] = batch * n_deep / (time.perf_counter() - t0)
                        deep[name + "_dma_batches"] = int(ctx.stats()["host_dma_batches"] - before)
                    deep["unit"] = UNIT
                    e2e["three_sets_two_batches_behind"] = deep
                except Exception as e:      # noqa: BLE001
                    e2e["three_sets_two_batches_behind"] = {"failed": repr(e)}
                finally:
                    ctx.set_host_dma(int(os.environ.get("FLUC_TTMLBLEND_HOST_DMA", "2")))
            # the same frames, one synchronous call per frame through the C mirror of the GStreamer
            # call (fluc_video_overlay_composition_blend == gst_video_overlay_composition_blend):
            # what a single streaming thread sees; not batched, so latency-bound
            try:
                vo = pkg.videooverlay
                if vo.load_library().fluc_video_overlay_set_device(local) == 0:
                    comp = vo.Composition(vo.Rectangle(work.overlay, 0, 0, vo.FLAG_PREMULTIPLIED_ALPHA))
                    views = [hf.host_planes() for hf in host_sets[0]]
                    for v in views[:4]:
                        comp.blend(fmt, W, H, v)
                    n_sync = 0
                    t0 = time.perf_counter()
                    while time.perf_counter() - t0 < 1.0:
                        comp.blend(fmt, W, H, views[n_sync % len(views)])
                        n_sync += 1
                    e2e["one_synchronous_call_per_frame"] = n_sync / (time.perf_counter() - t0)
                    del comp
            except Exception as e:      # noqa: BLE001
                e2e["one_synchronous_call_per_frame"] = f"failed: {e!r}"
            # ordinary (pageable) host memory: what an upstream element hands over when it does not
            # use the pinned allocator. No registration, no pinning behind the caller's back.
            try:
                n_pg = min(batch, 16)
                pg_frames = [[np.roll(p, i * 16, axis=1).copy() for p in base] for i in range(2 * n_pg)]
                F = pkg.ttmlblend._frame_from_arrays
                pg_c = [[F(f) for f in pg_frames[k * n_pg:(k + 1) * n_pg]] for k in range(2)]
                pgb = [ctx.Batch(stream_ids[:n_pg], fmt, W, H, c_, c_) for c_ in pg_c]

                def pageable_loop(n_steps):
                    prev = None
                    for i in range(n_steps):
                        t = ctx.blend_host_many(pgb[i & 1])
                        if prev is not None:
                            for x in prev:
                                ctx.wait(x)
                        prev = list(t)
                    for x in prev:
                        ctx.wait(x)

                pageable_loop(2)
                ctx.sync()
                n_p = max(4, min(e2e_steps, 20))
                t0 = time.perf_counter()
                pageable_loop(n_p)
                ctx.sync()
                e2e["pageable"] = {"value": n_pg * n_p / (time.perf_counter() - t0), "unit": UNIT,
                                   "frames_per_call": n_pg,
                                   "note": "numpy-allocated (pageable) frames, no host_register, no auto-register; "
                                           "this rank only"}
            except Exception as e:      # noqa: BLE001
                e2e["pageable"] = {"failed": repr(e)}
        for hs in host_sets:
            for hf in hs:
                hf.release()
        for f in work.srcs:
            f.release()
    else:
        work.release()

    # ---- BASELINE config 5 beside the headline: 256 streams sharded stream % N --------------
    cfg5 = None
    if extras and args.config == 3:
        try:
            c5 = wl.CONFIGS[5]
            w5 = DeviceWorkload(ctx, wl, sh, c5, c5.fmt, world, rank, stream_base=5000)
            ctx.set_batch(min(w5.batch, 1024), 0)
            w5.steps(args.warmup)
            ms5, st5 = timed_region(ctx, w5, args.steps, dist, device, profile_every)
            rec5 = sh.gather_records((w5.batch * args.steps, ms5), dist, device)
            rl5 = roofline_record(w5, ms5, st5, args.steps, peak, peak_src, c5.name, c5.fmt, kernel_name(c5.fmt))
            cfg5 = {"value": sh.aggregate_fps(rec5), "unit": UNIT, "scaling": "strong",
                    "streams": c5.streams, "streams_this_rank": w5.batch,
                    "ms_per_step": sh.reduce_max(ms5, dist, device) / args.steps,
                    "launches": int(st5["launches"]), "roofline": rl5,
                    "config": config_record(c5, wl, c5.fmt, world)}
            w5.release()
            for s_id in set(w5.stream_ids):
                ctx.overlay_clear(s_id)
            ctx.set_batch(min(batch, 1024), 0)
        except Exception as e:      # noqa: BLE001
            cfg5 = {"failed": repr(e)}

    # ---- several GPUs driven from ONE process (FlucTtmlBlendMulti), the other ranks idle ----
    multi = None
    if extras and world > 1 and cfg.streams == 1 and not args.no_e2e:
        gloo = dist.new_group(backend="gloo")
        barrier(dist, device)
        cpu_barrier(dist, gloo)
        if rank == 0:
            try:
                multi = run_multi_leg(pkg, wl, cfg, fmt, world, args.steps)
            except Exception as e:      # noqa: BLE001
                multi = {"failed": repr(e)}
        cpu_barrier(dist, gloo)
    sampler.stop()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = run_cpu_baseline(cfg, wl)

    if rank == 0:
        config = config_record(cfg, wl, fmt, world)
        line = {
            "metric": METRIC if args.config == 3 else f"frames/sec, TTML overlay blend ({cfg.name})",
            "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "warmup_extra_steps": warm_extra,
            "ms_per_step": worst_ms / args.steps, "higher_is_better": True,
            "scaling": work.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config,
            "steps_issued_by": "fluc_ttmlblend_submit_many_repeat: one native call runs the K steps "
                               "(a step = submit_many of the batch + flush = one launch)",
            "roofline": roofline, "sustained": sustained, "e2e": e2e, "cpu_baseline": cpu, "clocks": clocks,
            "gstreamer": ("present: " + shutil.which("gst-launch-1.0")) if shutil.which("gst-launch-1.0")
            else "absent on this box (no gst-launch-1.0): the reference pipeline itself cannot be timed",
            "gpu_launches": gpu_launches,
            "per_rank": [{"frames": r[0], "ms": r[1], "kernel_ms": r[2]} for r in records],
        }
        for k, v in (("inplace", inplace), ("distinct_cues", distinct), ("cfg5", cfg5), ("multi", multi)):
            if v is not None:
                line[k] = v
        print(json.dumps(line), file=real_stdout, flush=True)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


def run_multi_leg(pkg, wl, cfg, fmt, n_dev, steps):
    """Rank 0 drives all N GPUs from one process: one FlucTtmlBlendMulti, stream s on device s % N,
    device-resident batches and host-frame batches on every device from one thread."""
    W, H = cfg.width, cfg.height
    m = pkg.TtmlBlendMulti(list(range(n_dev)))
    try:
        ov = wl.overlay_for(cfg)
        base = wl.frame_for(cfg, 0, fmt)
        ctxs, dev_batches, host_batches, frames = [], [], [], []
        for s in range(n_dev):              # stream id s lives on device s
            c = m.context(s)
            c.overlay_set(s, ov, wl.region_rects(cfg))
            c.set_batch(cfg.batch, 0)
            srcs = [c.acquire(fmt, W, H) for _ in range(cfg.batch)]
            dsts = [c.acquire(fmt, W, H) for _ in range(cfg.batch)]
            for i, f in enumerate(srcs):
                f.upload([np.roll(p, i * 16, axis=1) for p in base])
            hsets = [[c.acquire(fmt, W, H, on_host=True) for _ in range(cfg.batch)] for _ in range(2)]
            for hs in hsets:
                for i, hf in enumerate(hs):
                    for dstp, srcp in zip(hf.host_planes(), base):
                        dstp[...] = np.roll(srcp, i * 16, axis=1)
            ctxs.append(c)
            dev_batches.append(c.Batch([s] * cfg.batch, fmt, W, H, [f.c for f in srcs], [f.c for f in dsts]))
            host_batches.append([c.Batch([s] * cfg.batch, fmt, W, H, [hf.c for hf in hs], [hf.c for hf in hs])
                                 for hs in hsets])
            frames.append((srcs, dsts, hsets))
        # device-resident: every device gets `steps` launches, issued round robin from this thread
        for c, b in zip(ctxs, dev_batches):
            c.submit_many(b)
        m.sync()
        for c in ctxs:
            c.timer_begin()
        for _ in range(steps):
            for c, b in zip(ctxs, dev_batches):
                c.submit_many(b)
        dev_ms = max(c.timer_end() for c in ctxs)
        m.sync()
        # host frames: the e2e loop, interleaved over the devices
        e2e_steps = max(4, min(steps, 40))

        def loop(n):
            prev = [None] * n_dev
            for i in range(n):
                for k, c in enumerate(ctxs):
                    t = c.blend_host_many(host_batches[k][i & 1])
                    if prev[k] is not None:
                        c.wait(prev[k])
                    prev[k] = t[len(t) - 1]
            for k, c in enumerate(ctxs):
                c.wait(prev[k])

        loop(16)                # long enough for every context to have tried both transports (see the e2e leg)
        m.sync()
        t0 = time.perf_counter()
        loop(e2e_steps)
        m.sync()
        dt = time.perf_counter() - t0
        return {"devices": n_dev, "value": n_dev * cfg.batch * steps / (dev_ms * 1e-3), "unit": UNIT,
                "e2e": n_dev * cfg.batch * e2e_steps / dt,
                "note": "one process, one thread, FlucTtmlBlendMulti over all N GPUs (stream s on device s % N) "
                        "while the other ranks wait at a barrier: device-resident batches (value; MAX of the "
                        "per-device timers) and pinned host frames (e2e; wall clock)"}
    finally:
        m.close()


if __name__ == "__main__":
    main()
