"""Measure several views of one resident scene in one call (Renderer.trace_views, tracer_cuda_render_views) against one
trace call per view, on one GPU, in one process.  Hash RNG, seed 42; the two routes alternate round by round (--rounds,
medians reported).

  A  soup_scene(100_000, 100, 4, seed=42) at 256x256, 64 eyes on a circle of radius 3 around (0, 1, 0) at height 1
  B  C4 (soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)) at 960x540, 16 eyes on the same circle
  C  C4 at 3840x2160, one view (0, 1, 3): trace against trace_views([cam])

Per route: the host clock around the whole route (ending in a device synchronise), the sum of the calls' ms_total and
its split (ms_primary, ms_shadow, ms_other; CUDA events).  Every view's sha256 must equal the single-view route's.  The
device name, power limit and max SM clock are read in the same run.

    python tools/views_bench.py [--rounds 5] [--out views_bench.txt] [--cases ABC]
"""
import argparse
import hashlib
import math
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from esctp1raytracer_b200 import RNG_HASH, Camera, Renderer, scenes  # noqa: E402


def gpu_query():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def circle_eyes(n):
    return [(3.0 * math.sin(2 * math.pi * i / n), 1.0, 3.0 * math.cos(2 * math.pi * i / n)) for i in range(n)]


def sha(a):
    return hashlib.sha256(a.tobytes()).hexdigest()


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--cases", default="ABC")
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("# python tools/views_bench.py " + " ".join(sys.argv[1:]))
    r = Renderer(0)
    info = r.device_info()
    say(f"device: {info['name']}, {info['sm_count']} SMs; nvidia-smi (name, power limit, max SM clock): {gpu_query()}")
    say(f"hash RNG, seed 42; routes alternated, medians of {a.rounds} rounds")
    c4 = None
    cases = []
    if "A" in a.cases:
        cases.append(("A", scenes.soup_scene(100_000, 100, 4, seed=42), 256, 256, circle_eyes(64)))
    if "B" in a.cases or "C" in a.cases:
        c4 = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    if "B" in a.cases:
        cases.append(("B", c4, 960, 540, circle_eyes(16)))
    if "C" in a.cases:
        cases.append(("C", c4, 3840, 2160, [(0.0, 1.0, 3.0)]))
    for name, scene, W, H, eyes in cases:
        rs = r.upload(scene)
        cams = [Camera.for_frame(e, (0, 1, 0), W, H) for e in eyes]

        def loop():
            return [r.trace(rs, c, W, H, rng_mode=RNG_HASH, seed=42) for c in cams]

        def batch():
            return r.trace_views(rs, cams, W, H, rng_mode=RNG_HASH, seed=42)

        ref = [sha(f.rgb8) for f in loop()]  # warm-up of both routes (tables, workspace)
        b = batch()
        same = all(sha(b.rgb8[v]) == ref[v] for v in range(len(cams)))
        res = {"loop": [], "batch": []}
        for _ in range(a.rounds):
            for route in ("loop", "batch"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = loop() if route == "loop" else batch()
                torch.cuda.synchronize()
                wall = (time.perf_counter() - t0) * 1e3
                stats = [f.stats for f in out] if route == "loop" else [out.stats]
                split = {k: sum(s[k] for s in stats) for k in ("ms_total", "ms_primary", "ms_shadow", "ms_other")}
                res[route].append(dict(wall=wall, **split))
                if route == "batch":
                    same &= all(sha(out.rgb8[v]) == ref[v] for v in range(len(cams)))
        say(f"case {name}: {len(cams)} view(s) of {W}x{H}, {scene.n_tris} triangles, {scene.n_lights} lights")
        for route in ("loop", "batch"):
            med = {k: statistics.median(x[k] for x in res[route]) for k in res[route][0]}
            label = f"{len(cams)} x trace" if route == "loop" else "1 x trace_views"
            say(f"  {label:16s} host {med['wall']:9.2f} ms   sum ms_total {med['ms_total']:9.2f}   ms_primary {med['ms_primary']:9.2f}"
                f"   ms_shadow {med['ms_shadow']:9.2f}   ms_other {med['ms_other']:8.2f}")
        lw = statistics.median(x["wall"] for x in res["loop"])
        bw = statistics.median(x["wall"] for x in res["batch"])
        say(f"  loop / batch (host clock): {lw / bw:.2f}x; every view's sha256 equals the single-view route's: {same}")
        rs.close()
        if not same:
            raise SystemExit("a view differs from its single render")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
