"""Scratch probe: blend pinned HOST frames in place through blend_host, the kernel reading and
writing them over PCIe directly (zero-copy). Config 3."""
import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import __graft_entry__ as graft
pkg = graft.load_package(); wl = pkg.workloads
cfg = wl.CONFIGS[3]
ctx = pkg.TtmlBlend(0)
ov = wl.overlay_for(cfg)
ctx.overlay_set(1, ov, wl.region_rects(cfg))
n = 32
hosts = [ctx.acquire(cfg.fmt, cfg.width, cfg.height, on_host=True) for _ in range(n)]
base = wl.frame_for(cfg, 0)
for hf in hosts:
    for d, s in zip(hf.host_planes(), base):
        d[...] = s
ctx.set_batch(n, 0)
def step_zc():
    t = [ctx.submit(1, cfg.fmt, cfg.width, cfg.height, hf.c, hf.c) for hf in hosts]
    ctx.wait(t[-1])
def step_host():
    t = [ctx.blend_host_frame(1, cfg.fmt, cfg.width, cfg.height, hf.c) for hf in hosts]
    for x in t: ctx.wait(x)
for name, fn in (("blend_host", step_host),):
    for _ in range(3): fn()
    ctx.sync(); t0 = time.perf_counter(); k = 30
    for _ in range(k): fn()
    ctx.sync(); dt = time.perf_counter() - t0
    print(f"{name}: {n*k/dt:.0f} frames/s  ({dt/k/n*1e6:.1f} us/frame)")
# correctness of zero-copy result vs oracle for one frame
from oracle import oracle
for hf in hosts[:1]:
    for d, s in zip(hf.host_planes(), base):
        d[...] = s
ctx.wait(ctx.submit(1, cfg.fmt, cfg.width, cfg.height, hosts[0].c, hosts[0].c))
want = oracle.composition_blend(cfg.fmt, cfg.width, cfg.height, [p.copy() for p in base], oracle.ttmlrender_rectangles(ov))
print("zero-copy bit-exact:", all(np.array_equal(a, b) for a, b in zip(hosts[0].host_planes(), want)))
