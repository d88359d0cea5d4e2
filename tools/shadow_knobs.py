"""Shadow-sweep knobs at C4 (profiles/r05_d): renders the C4 scene with Renderer.trace(shadow_chunks=c) for each c, one
warm-up and 3 timed frames, and prints the median/min/max of the library's shadow-sweep time (CUDA events), the median
closest-hit time and the frame hashes.  Env knobs (TRACER_RUN_PAIRS, TRACER_ITEMS_PER_CTA) are read by the library.

    python tools/shadow_knobs.py <repository root> <chunks,chunks,...> <tag>
"""
import hashlib, os, statistics, sys
root = sys.argv[1]; chunks = [int(x) for x in sys.argv[2].split(",")]; tag = sys.argv[3]
sys.path.insert(0, root)
from esctp1raytracer_b200 import Renderer, Camera, scenes
s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
W, H = 3840, 2160
cam = Camera.for_frame((0.0, 1.0, 3.0), (0.0, 1.0, 0.0), W, H)
r = Renderer(0); rs = r.upload(s)
for c in chunks:
    r.trace(rs, cam, W, H, seed=42, shadow_chunks=c)
    sh, pr, h = [], [], set()
    for _ in range(3):
        o = r.trace(rs, cam, W, H, seed=42, shadow_chunks=c)
        sh.append(o.stats["ms_shadow"]); pr.append(o.stats["ms_primary"]); h.add(hashlib.sha256(o.rgb8.tobytes()).hexdigest()[:16])
    print("KNOB", tag, "chunks", c, "shadow med %.2f min %.2f max %.2f" % (statistics.median(sh), min(sh), max(sh)), "prim %.2f" % statistics.median(pr), h, flush=True)
