"""Measure resident-scene updates (ResidentScene.update, tracer_cuda_scene_update) against re-creating the scene, on one
GPU, in one process.

C4: soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42), 3840x2160, hash RNG, seed 42.  Cases, in the default and
bundle-cull modes, alternated round by round (--rounds, medians reported):
  plain        a resident frame, nothing changed
  geom_np      one geometry (geometry 500, about 1000 triangles) moved, from numpy
  geom_torch   the same, from a torch CUDA tensor
  all_np       every triangle moved (translated by 0.02 in x), from numpy
  all_torch    the same, from a torch CUDA tensor
  light        light 0's quad moved, from numpy
  recreate     destroy, create from numpy and a first frame (the route without updates)
and, in the BVH mode, plain (kept tree) and geom_np (the first BVH frame after an update rebuilds the tree).
Per case: the update call (host clock around the synchronous call; for recreate: destroy + create), and the next frame's
ms_total and ms_other (CUDA events; ms_other holds the rebuilt tree in the BVH mode, while the lazily rebuilt shadow
tables are timed inside the shadow sweeps' window).  After each timed
case the scene is updated back and one untimed frame per mode restores the steady state.  Every updated frame's sha256 must equal
the frame of a freshly created scene of the same arrays.  The device name, power limit and max SM clock are read in the
same run.

    python tools/scene_update_bench.py [--rounds 5] [--out scene_update_bench.txt]
"""
import argparse
import hashlib
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from esctp1raytracer_b200 import RNG_HASH, Camera, Renderer, Scene, scenes  # noqa: E402


def gpu_query():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    r = Renderer(0)
    info = r.device_info()
    say(f"device: {info['name']}, {info['sm_count']} SMs; nvidia-smi name, power limit, max SM clock: {gpu_query()}")
    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    o = s.geom_tri_offset
    g0, g1 = int(o[500]), int(o[501])
    l0, l1 = int(o[1]), int(o[2])
    v = s.tri_verts
    geom_new = v[g0:g1].copy()
    c = geom_new.mean(axis=1, keepdims=True)
    geom_new = (np.array([0.0, 1.3, 0.6], np.float32) + (c - c.mean(axis=0)) * np.float32(0.3) + (geom_new - c) * np.float32(3.0)).astype(np.float32)
    all_new = (v + np.array([0.02, 0.0, 0.0], np.float32)).astype(np.float32)
    light_new = (v[l0:l1] + np.array([0.1, -0.05, 0.05], np.float32)).astype(np.float32)
    geom_t, all_t = torch.from_numpy(geom_new).cuda(), torch.from_numpy(all_new).cuda()
    torch.cuda.synchronize()
    say(f"scene: {s.n_tris} triangles, {s.n_geoms} geometries, {s.n_lights} lights, {len(s.sphere_cr)} spheres; {W}x{H}; "
        f"one geometry = triangles [{g0}, {g1}) ({g1 - g0}); light 0 = triangles [{l0}, {l1})")

    def replaced(first, new):
        w = v.copy()
        w[first:first + len(new)] = new
        return w

    # case -> (update kwargs, restore kwargs, the updated vertex array for the fresh-scene hash)
    cases = {
        "plain": None,
        "geom_np": (dict(tri_verts=geom_new, first_tri=g0), dict(tri_verts=v[g0:g1], first_tri=g0), replaced(g0, geom_new)),
        "geom_torch": (dict(tri_verts=geom_t, first_tri=g0), dict(tri_verts=v[g0:g1], first_tri=g0), None),
        "all_np": (dict(tri_verts=all_new), dict(tri_verts=v), all_new),
        "all_torch": (dict(tri_verts=all_t), dict(tri_verts=v), None),
        "light": (dict(tri_verts=light_new, first_tri=l0), dict(tri_verts=v[l0:l1], first_tri=l0), replaced(l0, light_new)),
        "recreate": "recreate",
    }
    want_hash = {}
    sha = lambda f: hashlib.sha256(f.rgb8.tobytes()).hexdigest()
    for name, cdef in cases.items():  # the fresh scenes' frames
        if isinstance(cdef, tuple) and cdef[2] is not None:
            fresh = r.upload(Scene(s.geom_tri_offset, cdef[2], s.geom_material, s.light_geom, sphere_cr=s.sphere_cr,
                                          sphere_material=s.sphere_material))
            want_hash[name] = sha(r.trace(fresh, cam, W, H, rng_mode=RNG_HASH, seed=seed))
            fresh.close()
    want_hash["geom_torch"], want_hash["all_torch"] = want_hash["geom_np"], want_hash["all_np"]
    rs = r.upload(s)
    base_hash = sha(r.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed))
    want_hash["plain"] = want_hash["recreate"] = base_hash
    say(f"frame sha256: unchanged {base_hash[:16]}..., one geometry {want_hash['geom_np'][:16]}..., all {want_hash['all_np'][:16]}..., "
        f"light {want_hash['light'][:16]}...")
    modes = {"default": {}, "bundle_cull": dict(bundle_cull=True), "bvh": dict(bvh=True)}
    mode_cases = {"default": list(cases), "bundle_cull": list(cases), "bvh": ["plain", "geom_np"]}
    for m in modes.values():  # warm-up: every mode's tables / tree built
        r.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, **m)
    res = {(m, c): [] for m in modes for c in mode_cases[m]}
    mismatches = []
    for rnd in range(a.rounds):
        for mname, mkw in modes.items():
            for cname in mode_cases[mname]:
                cdef = cases[cname]
                t0 = time.perf_counter()
                if cdef == "recreate":
                    rs.close()
                    rs = r.upload(s)
                elif cdef is not None:
                    rs.update(**cdef[0])
                t_upd = (time.perf_counter() - t0) * 1e3
                f = r.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, **mkw)
                if sha(f) != want_hash[cname]:
                    mismatches.append((rnd, mname, cname))
                res[(mname, cname)].append((t_upd if cdef is not None else 0.0, f.stats["ms_total"], f.stats["ms_other"]))
                if isinstance(cdef, tuple):
                    rs.update(**cdef[1])
                if cdef is not None:  # back to the steady state of every mode before the next case
                    for m in modes.values():
                        r.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, **m)
    say(f"medians of {a.rounds} alternated rounds; update = host clock around the synchronous call (recreate: destroy + create "
        "from numpy); ms_total / ms_other = CUDA events of the next frame")
    say(f"{'mode':<12} {'case':<11} {'update ms':>10} {'frame ms_total':>15} {'ms_other':>9}   (min-max of ms_total)")
    for (mname, cname), xs in res.items():
        med = [statistics.median(x[i] for x in xs) for i in range(3)]
        tot = [x[1] for x in xs]
        say(f"{mname:<12} {cname:<11} {med[0]:10.2f} {med[1]:15.2f} {med[2]:9.2f}   ({min(tot):.2f}-{max(tot):.2f})")
    say("every updated frame's sha256 equals the fresh scene's: " + ("yes" if not mismatches else f"NO: {mismatches}"))
    rs.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    return 1 if mismatches else 0


if __name__ == "__main__":
    sys.exit(main())
