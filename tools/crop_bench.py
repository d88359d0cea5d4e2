"""Measure crop windows (Renderer.trace(..., crop=...)) against the whole frame on one GPU, in one process: C4
(soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)) at 3840x2160, eye (0, 1, 3), seed 42.

Windows (x, y, w, h in PPM coordinates):
  centre     256 x 256 in the middle of the frame
  corner     512 x 512 at the bottom right: with seeded faceIDs its covering rows are the whole frame (the worst case)
  row        one full-width row in the middle
each in hash (RNG_HASH) and seeded (RNG_MT19937) mode, in the default sweeps and the bundle-cull mode (bundle_cull=1).

Per (mode, RNG mode) the whole frame and the three windows alternate round by round (--rounds, medians reported): the host
clock around the call (it ends in a device synchronise) and the call's ms_total with its split (ms_primary, ms_shadow,
ms_other; CUDA events).  Every window's sha256 must equal that of the same window cut from the whole frame.  The device
name, power limit and max SM clock are read in the same run.

    python tools/crop_bench.py [--rounds 3] [--out crop_bench.txt]
"""
import argparse
import hashlib
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from esctp1raytracer_b200 import RNG_HASH, RNG_MT19937, Camera, Renderer, scenes  # noqa: E402

W, H = 3840, 2160
WINDOWS = {"centre": ((W - 256) // 2, (H - 256) // 2, 256, 256), "corner": (W - 512, H - 512, 512, 512), "row": (0, H // 2, W, 1)}


def gpu_query():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def sha(a):
    return hashlib.sha256(a.tobytes()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("# python tools/crop_bench.py " + " ".join(sys.argv[1:]))
    r = Renderer(0)
    info = r.device_info()
    say(f"device: {info['name']}, {info['sm_count']} SMs; nvidia-smi (name, power limit, max SM clock): {gpu_query()}")
    scene = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    say(f"C4: {scene.n_tris} triangles, {len(scene.sphere_cr)} spheres, {scene.n_lights} lights, {W}x{H}, seed 42; "
        f"whole frame and windows alternated, medians of {a.rounds} rounds")
    rs = r.upload(scene)
    cam = Camera.for_frame((0.0, 1.0, 3.0), (0.0, 1.0, 0.0), W, H)
    ok = True
    for mode_name, mode in (("default", {}), ("bundle-cull", dict(bundle_cull=1))):
        for rng_name, rng in (("hash", RNG_HASH), ("seeded", RNG_MT19937)):
            kw = dict(rng_mode=rng, seed=42, **mode)
            routes = {"frame": None, **WINDOWS}

            def run(window):
                t0 = time.perf_counter()
                f = r.trace(rs, cam, W, H, crop=window, **kw)  # returns after the read-back's synchronise
                return f, (time.perf_counter() - t0) * 1e3

            full, _ = run(None)  # warm-up: tables, workspace
            want = {k: sha(full.rgb8[w[1]:w[1] + w[3], w[0]:w[0] + w[2]]) for k, w in WINDOWS.items()}
            for window in WINDOWS.values():
                run(window)
            res = {k: [] for k in routes}
            same = True
            for _ in range(a.rounds):
                for k, window in routes.items():
                    f, wall = run(window)
                    res[k].append(dict(wall=wall, **{s: f.stats[s] for s in ("ms_total", "ms_primary", "ms_shadow", "ms_other")}))
                    if window is not None:
                        same &= sha(f.rgb8) == want[k]
                    else:
                        same &= sha(f.rgb8) == sha(full.rgb8)
            say(f"{mode_name}, {rng_name}:")
            frame_ms = statistics.median(x["ms_total"] for x in res["frame"])
            for k, window in routes.items():
                med = {s: statistics.median(x[s] for x in res[k]) for s in res[k][0]}
                label = f"{W}x{H} frame" if window is None else f"{k} {window[2]}x{window[3]} @ ({window[0]}, {window[1]})"
                say(f"  {label:32s} host {med['wall']:8.2f} ms   ms_total {med['ms_total']:8.2f} ({med['ms_total'] / frame_ms:6.1%} of the frame)"
                    f"   ms_primary {med['ms_primary']:7.2f}   ms_shadow {med['ms_shadow']:7.2f}   ms_other {med['ms_other']:6.2f}")
            say(f"  every window's sha256 equals the whole frame's window: {same}")
            ok &= same
    rs.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    if not ok:
        raise SystemExit("a window differs from the whole frame")


if __name__ == "__main__":
    main()
