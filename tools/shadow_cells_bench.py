"""Shadow sweeps at C4 with the rays ordered in (p, q) cells (profiles/r11_*): renders the C4 scene (1 M triangles + 1 k
spheres, 3840x2160, 4 lights, default mode) with Renderer.trace(shadow_chunks=c) for each c, one warm-up and N timed frames,
and prints per setting the median/min/max of the frame time (ms_total) and of the shadow-sweep time (ms_shadow, CUDA events),
the median closest-hit time, the frame hashes and, with TRACER_SHADOW_DIAG=1 in the environment, the library's diagnostic
line of the last frame (flagged (thread, triangle) verdicts, queued pairs, strict evaluations, the item/barrier/compaction
split).  --profile adds one frame under torch.profiler and prints the kernel time of the shadow-ray ordering
(order_shadow_rays: the radix sorts, stripe_key_kernel, list_prefix_kernel).  The stripe length is the library's
TRACER_SHADOW_STRIPE (unset: each group's own, from SHADOW_CELL_C in kernels.cuh), so a stripe sweep is one process per value.

    python tools/shadow_cells_bench.py <repository root> <tag> [--chunks 32,48] [--frames 3] [--profile]
"""
import argparse, hashlib, os, statistics, sys

ap = argparse.ArgumentParser()
ap.add_argument("root")
ap.add_argument("tag")
ap.add_argument("--chunks", default="0", help="shadow_chunks values; 0 = the library's default")
ap.add_argument("--frames", type=int, default=3)
ap.add_argument("--profile", action="store_true")
args = ap.parse_args()
knobs = {k: v for k, v in os.environ.items() if k.startswith("TRACER_")}
print("CMD", " ".join([os.path.basename(sys.executable)] + sys.argv), knobs, flush=True)
sys.path.insert(0, args.root)
from esctp1raytracer_b200 import Camera, Renderer, scenes  # noqa: E402

s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
W, H = 3840, 2160
cam = Camera.for_frame((0.0, 1.0, 3.0), (0.0, 1.0, 0.0), W, H)
r = Renderer(0)
rs = r.upload(s)
for c in [int(x) for x in args.chunks.split(",")]:
    r.trace(rs, cam, W, H, seed=42, shadow_chunks=c)
    tot, sh, pr, h = [], [], [], set()
    for _ in range(args.frames):
        sys.stderr.flush()
        o = r.trace(rs, cam, W, H, seed=42, shadow_chunks=c)
        tot.append(o.stats["ms_total"]), sh.append(o.stats["ms_shadow"]), pr.append(o.stats["ms_primary"])
        h.add(hashlib.sha256(o.rgb8.tobytes()).hexdigest()[:16])
    st = o.stats
    print("RESULT", args.tag, "chunks", c, "total med %.2f min %.2f max %.2f" % (statistics.median(tot), min(tot), max(tot)),
          "shadow med %.2f min %.2f max %.2f" % (statistics.median(sh), min(sh), max(sh)), "prim %.2f" % statistics.median(pr),
          "strict", st["strict_evals"], "tests_shadow", st["tests_shadow"], "launches", st["kernel_launches"], sorted(h), flush=True)
if args.profile:
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r.trace(rs, cam, W, H, seed=42)
        torch.cuda.synchronize()
    order, rest = {}, 0.0
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if any(x in e.key for x in ("RadixSort", "Onesweep", "stripe_key_kernel", "list_prefix_kernel")):
            order[e.key[:60]] = (e.count, us / 1e3)
        else:
            rest += us / 1e3
    print("ORDER", args.tag, "ms %.3f" % sum(v[1] for v in order.values()), {k: (n, round(ms, 3)) for k, (n, ms) in order.items()},
          "other kernels ms %.1f" % rest, flush=True)
