"""Measure the seeded std::mt19937 mode (RNG_MT19937), whose draws are replayed on the device, against the hash mode.

C4 (bench.py's configuration): soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42), 3840x2160, resident scene, seed 42.
* seeded and hash frames alternated after a warm-up frame each, --frames of each: the library's CUDA-event frame time
  (ms_total: the replay's host steps, a read-back of the row counts and of the stream's hit count, are inside it) and the
  host wall time of the call;
* the device replay on its own (tracer__mt19937_faceids_device on the frame's hit mask: CUDA events from the per-row hit
  count to the gather) and its stream generator on its own (tracer__mt19937_stream_device: events around the launch),
  against tracer_mt19937_faceids on the same mask in the same process: the serial host work the replay replaces, before
  its copies;
* the seeded frame's sha256 against the frame rendered from tracer_mt19937_faceids' faceIDs (RNG_EXPLICIT);
* with two or more GPUs: seeded against hash frames on all of them (MultiRenderer, host wall time).
The device name and power limit are read in the same run.

    python tools/mt19937_bench.py [--frames 3] [--out profiles/r06_a_mt19937_bench.txt]
"""
import argparse
import ctypes as C
import hashlib
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bvh_bench import power_limit  # noqa: E402

from esctp1raytracer_b200 import (RNG_EXPLICIT, RNG_HASH, RNG_MT19937, Camera, MultiRenderer, Renderer, _lib,  # noqa: E402
                                  mt19937_faceids, scenes)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    r = Renderer(0)
    lib = _lib.load()
    lib.tracer__mt19937_faceids_device.argtypes = [C.c_uint32, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_int32,
                                                   C.POINTER(C.c_uint8), C.POINTER(C.c_int32), C.POINTER(C.c_double)]
    info = r.device_info()
    say(f"device: {info['name']}, {info['sm_count']} SMs; nvidia-smi name, power limit, max SM clock: {power_limit()}")
    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = r.upload(s)
    sha = lambda f: hashlib.sha256(f.rgb8.tobytes()).hexdigest()  # noqa: E731

    dbg = r.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=seed, debug=True)
    hit_img = np.ascontiguousarray(dbg.tri.reshape(H, W)[::-1] >= 0).reshape(-1)
    t0 = time.perf_counter()
    fid = mt19937_faceids(s, W, H, seed, hit_img)
    host_ms = (time.perf_counter() - t0) * 1e3
    want = sha(r.trace(rs, cam, W, H, rng_mode=RNG_EXPLICIT, faceid=fid))

    modes = {"seeded": RNG_MT19937, "hash": RNG_HASH}
    res = {m: [] for m in modes}
    shas = {m: sha(r.trace(rs, cam, W, H, rng_mode=mode, seed=seed)) for m, mode in modes.items()}  # warm-up
    for _ in range(a.frames):
        for m, mode in modes.items():
            t0 = time.perf_counter()
            f = r.trace(rs, cam, W, H, rng_mode=mode, seed=seed)
            res[m].append((f.stats["ms_total"], (time.perf_counter() - t0) * 1e3))
            assert sha(f) == shas[m]
    say(f"C4 3840x2160, 1M triangles + 1k spheres, 4 lights, seed 42, {int(hit_img.sum())} hit pixels; {a.frames} frames of "
        "each mode, alternated, after a warm-up frame each")
    med = {m: (float(np.median([x[0] for x in v])), float(np.median([x[1] for x in v]))) for m, v in res.items()}
    for m in modes:
        say(f"  {m:7s} ms_total {med[m][0]:8.2f} (median of {[round(x[0], 2) for x in res[m]]})  host wall {med[m][1]:8.2f} ms")
    diff = med["seeded"][0] - med["hash"][0]

    scan = np.ascontiguousarray(hit_img.reshape(H, W)[::-1]).reshape(-1).astype(np.uint8)
    faces = np.asarray(s.faces_per_light, np.int32)
    dev_ms = []
    for _ in range(3):
        out = np.empty((W * H, len(faces)), np.int32)
        ms = C.c_double()
        _lib.check(lib.tracer__mt19937_faceids_device(seed, len(faces), faces.ctypes.data_as(C.POINTER(C.c_int32)), W, H,
                                                      scan.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                      out.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(ms)))
        dev_ms.append(ms.value)
        assert np.array_equal(out.reshape(H, W, -1)[::-1].reshape(W * H, -1), fid)
    say(f"  device replay alone: {float(np.median(dev_ms)):.2f} ms (median of {[round(x, 2) for x in dev_ms]}), faceIDs equal "
        "tracer_mt19937_faceids'")
    lib.tracer__mt19937_stream_device.argtypes = [C.c_uint32, C.c_int64, C.POINTER(C.c_double)]
    n_words = 3 * len(faces) * int(hit_img.sum())
    gen_ms = []
    for _ in range(3):
        ms = C.c_double()
        _lib.check(lib.tracer__mt19937_stream_device(seed, n_words, C.byref(ms)))
        gen_ms.append(ms.value)
    say(f"  of which the stream generator alone ({n_words} words, one CTA, CUDA events around its launch): "
        f"{float(np.median(gen_ms)):.2f} ms (median of {[round(x, 2) for x in gen_ms]})")
    say(f"  host replay (tracer_mt19937_faceids, same mask, same process): {host_ms:.1f} ms")
    say(f"  seeded - hash frame time: {diff:.2f} ms; below the host replay: {diff < host_ms}")
    say(f"  seeded frame sha256 {shas['seeded'][:16]}, from tracer_mt19937_faceids + RNG_EXPLICIT {want[:16]}: equal {shas['seeded'] == want}")
    rs.close()

    import torch

    n = torch.cuda.device_count()
    if n < 2:
        say("  N GPUs: not measured (one GPU visible)")
    else:
        m = MultiRenderer(n)
        ms_ = m.upload(s)
        one = {md: sha(m.trace(ms_, cam, W, H, rng_mode=mode, seed=seed)) for md, mode in modes.items()}
        wall = {md: [] for md in modes}
        for _ in range(a.frames):
            for md, mode in modes.items():
                t0 = time.perf_counter()
                f = m.trace(ms_, cam, W, H, rng_mode=mode, seed=seed)
                wall[md].append((time.perf_counter() - t0) * 1e3)
                assert sha(f) == one[md]
        say(f"  {n} GPUs (MultiRenderer, host wall, median of {a.frames}): seeded {np.median(wall['seeded']):.2f} ms, hash "
            f"{np.median(wall['hash']):.2f} ms; seeded frame equals the 1-GPU frame: {one['seeded'] == shas['seeded']}")
        ms_.close()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
