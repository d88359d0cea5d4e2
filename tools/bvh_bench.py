"""Measure the optional BVH mode against the default and bundle-cull modes on one GPU, in one process.

C4: soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42), 3840x2160, hash RNG, seed 42, resident scene.  The three
modes are alternated after a warm-up frame each, --frames timed frames per mode; per mode the library's CUDA-event split
(ms_total / primary / shadow / other), the sha256 of the frame (all three must agree) and the strict tests per ray.  The
tree's build is timed on its own (tracer__bvh_prepare: CUDA events around the build, then a synchronise).  The share of
the spheres' brute-force loop is measured by rendering the same scene without its spheres.  Then an N sweep in BVH mode
at 1920x1080.  The device name and power limit are read in the same run.

    python tools/bvh_bench.py [--frames 5] [--out profiles/r03_c_bvh_bench.txt]
"""
import argparse
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from esctp1raytracer_b200 import RNG_HASH, Camera, Renderer, _lib, scenes  # noqa: E402


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    r = Renderer(0)
    lib = _lib.load()
    lib.tracer__bvh_prepare.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    info = r.device_info()
    say(f"device: {info['name']}, {info['sm_count']} SMs; nvidia-smi name, power limit, max SM clock: {power_limit()}")

    def build_ms(rs):
        ms = C.c_double()
        _lib.check(lib.tracer__bvh_prepare(rs.handle, C.byref(ms)))
        return ms.value

    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = r.upload(s)
    modes = {"default": {}, "bundle_cull": dict(bundle_cull=True), "bvh": dict(bvh=True)}
    res = {m: [] for m in modes}
    sha = {}
    for m, kw in modes.items():  # warm-up (the BVH frame builds the tree)
        f = r.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, **kw)
        sha[m] = hashlib.sha256(f.rgb8.tobytes()).hexdigest()
    for _ in range(a.frames):
        for m, kw in modes.items():
            f = r.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, **kw)
            res[m].append(f.stats)
            assert hashlib.sha256(f.rgb8.tobytes()).hexdigest() == sha[m]
    say(f"C4 3840x2160, 1M triangles + 1k spheres, 4 lights, hash RNG seed 42; {a.frames} timed frames per mode, alternated")
    for m in modes:
        st = res[m]
        med = {k: float(np.median([x[k] for x in st])) for k in ("ms_total", "ms_primary", "ms_shadow", "ms_other")}
        rays = st[-1]["n_primary_rays"] + st[-1]["n_shadow_rays"]
        say(f"  {m:12s} ms_total {med['ms_total']:9.2f}  primary {med['ms_primary']:9.2f}  shadow {med['ms_shadow']:9.2f}  "
            f"other {med['ms_other']:7.2f}  (median; min total {min(x['ms_total'] for x in st):.2f})  "
            f"strict tests/ray {st[-1]['strict_evals'] / rays:10.1f}  tests/ray {(st[-1]['tests_primary'] + st[-1]['tests_shadow']) / rays:12.1f}"
            f"  sha256 {sha[m][:16]}")
    say(f"  frame sha256 equal in all three modes: {len(set(sha.values())) == 1}")
    bms = [build_ms(rs) for _ in range(3)]
    say(f"  BVH build (1M triangles, own call, CUDA events + synchronise): {' / '.join(f'{x:.2f}' for x in bms)} ms")
    s0 = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=0, seed=42)
    rs0 = r.upload(s0)
    r.trace(rs0, cam, W, H, rng_mode=RNG_HASH, seed=seed, bvh=True)
    no_sph = [r.trace(rs0, cam, W, H, rng_mode=RNG_HASH, seed=seed, bvh=True).stats for _ in range(a.frames)]
    tot0 = float(np.median([x["ms_total"] for x in no_sph]))
    tot1 = float(np.median([x["ms_total"] for x in res["bvh"]]))
    say(f"  spheres: the same frame without its 1000 spheres takes {tot0:.2f} ms in BVH mode (primary "
        f"{np.median([x['ms_primary'] for x in no_sph]):.2f}, shadow {np.median([x['ms_shadow'] for x in no_sph]):.2f}): "
        f"the spheres' brute-force loops cost ~{tot1 - tot0:.2f} ms of {tot1:.2f}")
    del rs0, rs
    say("N sweep, BVH mode, 1920x1080, soup_scene(N, 1000, 4, seed=42), no spheres (median of 3 frames after a warm-up)")
    cam2 = Camera.for_frame((0, 1, 3), (0, 1, 0), 1920, 1080)
    for n in (10_000, 100_000, 1_000_000, 4_000_000):
        sn = scenes.soup_scene(n, 1000, 4, seed=42)
        rsn = r.upload(sn)
        b = build_ms(rsn)
        r.trace(rsn, cam2, 1920, 1080, rng_mode=RNG_HASH, seed=seed, bvh=True)
        st = [r.trace(rsn, cam2, 1920, 1080, rng_mode=RNG_HASH, seed=seed, bvh=True).stats for _ in range(3)]
        rays = st[-1]["n_primary_rays"] + st[-1]["n_shadow_rays"]
        say(f"  N {n:>9d}: ms_total {np.median([x['ms_total'] for x in st]):8.2f}  primary {np.median([x['ms_primary'] for x in st]):8.2f}  "
            f"shadow {np.median([x['ms_shadow'] for x in st]):8.2f}  build {b:7.2f} ms  strict tests/ray {st[-1]['strict_evals'] / rays:8.1f}")
        del rsn
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
