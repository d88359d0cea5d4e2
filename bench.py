#!/usr/bin/env python
"""bench.py — the reference's headline metric on BASELINE.json's config.

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus N --native-dist ...               (ours, ONE process driving N GPUs through the C ABI)
    python bench.py ... --dump-outputs DIR                   (also write the last timed frame to DIR/*.npy)

Metric: Mrays/s (primary + shadow rays of one frame / frame time).  A "step" is one frame
of the hot path over synthetic input.  Default workload = BASELINE.json configs[3]:
synthetic 1M-triangle + 1k-sphere scene at 3840x2160, 4 lights ("c4").  Other workloads
(--workload c1|c3|c5|small) are development conveniences, not bench lines.

`value`  : scene resident in HBM, frame left in HBM on rank 0 (CUDA events, max over ranks).
`e2e`    : N = 1: the literal drop-in call tracer_cuda_render(scene, camera, W, H, opts, rgb_out) with HOST buffers
           every step — pinned host scene -> HBM, filter-table build, render, packed frame -> pinned host.
           N > 1: per rank scene upload + render + band gather, rank 0 reads the assembled frame back.
`roofline`: FP32-FMA bound (no tensor cores on this path).  achieved = FP32 flops the sweeps' formulation needs per
           (ray, triangle) pair (all in the FMA pipe, reported by the library: span form 4 + 8/R) x ALGORITHMIC pairs
           (P*N primary + the reference's own in-order count for shadow rays) / sweep-kernel time; peak = our own FFMA
           microbenchmark measured in the same process (MEASURED_PEAKS.json has no FP32 number).  Beside it: the nominal
           peak, the ceiling of this instruction mix, the as-issued flop count and the FMA-pipe lane-op utilisation.
`cpu_baseline`: the UNMODIFIED reference compiled from /root/reference (kind "reference"; oracle/_ref_release =
           its own Release flags -O3 -ffast-math for timing, oracle/_ref = strict build beside it) or the plain-C
           port, on a bounded pixel sample of the same workload; plus serial-1-core, the reference's --thread scheme,
           an AVX2 restatement, and "ispc": n/a.
`frame_sha256`: SHA-256 of the assembled frame on rank 0 (default mode and, when measured, bundle-cull mode): must
           be the same string for every N.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_PAIR = 12.0      # 6 FFMA (2-D affine edge rows) per (ray, triangle) pair when every ray evaluates its own rows
FLOP_PER_PAIR_REF = 46.0  # Moller-Trumbore with precomputed edges (SURVEY 8d), reported beside it
EYE, LOOK = (0.0, 1.0, 3.0), (0.0, 1.0, 0.0)

WORKLOADS = {
    # name: (n_tris, n_geoms, n_lights, n_spheres, W, H)
    "c4": (1_000_000, 1000, 4, 1000, 3840, 2160),
    "c3": (7_088, 9, 1, 0, 1920, 1080),       # CornellBox-Water as loaded by the reference (tests/golden/cornell_water.npz)
    "c1": (36, 7, 1, 0, 1024, 768),           # CornellBox-Original, the reference's default run (tests/golden/cornell_original.npz)
    "small": (100_000, 100, 4, 100, 1280, 720),
    # BASELINE.json configs[4]: 7680x4320, 16 spp jittered primary rays, 1 light, triangle-count sweep via --tris
    # (extension, parity unpinned; not a bench line: run with --workload c5 --tris N [--mode cull])
    "c5": (1_000_000, 1000, 1, 0, 7680, 4320),
}
WORKLOAD_SPP = {"c5": 16}
GOLDEN_MODELS = {"c1": "cornell_original.npz", "c3": "cornell_water.npz"}
DUMP_BYTES = 64 << 20   # --dump-outputs writes at most this much
DUMP_SAMPLE_PIXELS = 1 << 21


def dump_outputs(out_dir, frame):
    """Write the frame [H, W, 3] (uint8, PPM row order) of the last timed step as float32 .npy files: whole as
    frame.npy when it fits DUMP_BYTES, else a fixed seeded sample of DUMP_SAMPLE_PIXELS pixels as frame_sample.npy
    [k, 3] beside their flat pixel indices (h * W + w in PPM row order) as frame_sample_pixel.npy (float64, exact)."""
    os.makedirs(out_dir, exist_ok=True)
    rgb = np.asarray(frame).reshape(-1, 3)
    if rgb.size * 4 <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "frame.npy"), np.asarray(frame, np.float32))
        return
    idx = np.sort(np.random.default_rng(0).choice(len(rgb), DUMP_SAMPLE_PIXELS, replace=False))
    np.save(os.path.join(out_dir, "frame_sample.npy"), rgb[idx].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_sample_pixel.npy"), idx.astype(np.float64))


def make_scene(name, args):
    from esctp1raytracer_b200 import scenes  # pure numpy: does not load the CUDA library

    n_tris, n_geoms, n_lights, n_spheres, W, H = WORKLOADS[name]
    n_tris = args.tris or n_tris
    W, H = args.width or W, args.height or H
    if name in GOLDEN_MODELS and not args.tris:
        global EYE, LOOK
        sc, EYE, LOOK = scenes.from_npz(os.path.join(ROOT, "tests", "golden", GOLDEN_MODELS[name]))
        return sc, W, H
    return scenes.soup_scene(n_tris, min(n_geoms, max(8, n_tris // 100)), n_lights, n_spheres=n_spheres, seed=42), W, H


def workload_config(name, scene, W, H, spp, mode):
    """identical for both arms (the driver compares the `config` objects of `ours` and `reference`)"""
    kind = f"reference model {GOLDEN_MODELS[name][:-4]}" if name in GOLDEN_MODELS and scene.n_tris == WORKLOADS[name][0] else "synthetic"
    return {"workload": f"{name}: {kind} {scene.n_tris}-triangle + {len(scene.sphere_cr)}-sphere scene at {W}x{H}, "
                        f"{scene.n_lights} lights, brute force over all objects",
            "n_tris": scene.n_tris, "n_spheres": int(len(scene.sphere_cr)), "width": W, "height": H,
            "n_lights": scene.n_lights, "spp": max(1, spp), "mode": mode,
            "l2_policy": "working set larger than L2, no explicit flush: every step rewrites and re-reads its per-pixel ray "
            "workspace (~130 B/pixel: >= 1 GB per 4K frame on one GPU, >= 135 MB per GPU at 8) against a 126 MB L2, so "
            "nothing of step k is still cached at step k+1; the 32 MB span table is L2-resident WITHIN a step by design (it "
            "is swept by every ray block) and is rebuilt from the vertices every frame in the e2e path; no cached outputs",
            "rng": "counter-based hash (seeded)", "partition": "interleaved 8-row bands, scene replicated",
            "spheres": "analytic spheres are an extension the reference does not have: the GPU arm renders them, the CPU "
                       "reference arm cannot (it renders the same triangles and lights without them)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines, self.first = gpu_index, None, [], 0

    def mark(self):
        """the timed region starts here: only samples that arrive from now on are reported"""
        self.first = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for l in (self.lines[self.first:] or self.lines):  # (a region shorter than one sampling period: all samples)
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm.  Nothing here touches libtracer_cuda.so: scenes / hash_faceids are numpy, the camera comes from the oracle.
def cpu_sample(scene, W, H, n_pixels, threads, seed=42, extras=False):
    """Time the reference's own CPU path on a pixel sample of this workload."""
    from esctp1raytracer_b200.api import hash_faceids  # numpy mirror of the device hash; no library call
    from oracle import FlatScene, RefOracle, Restated, ref_available, ref_release_available

    rng = np.random.default_rng(7)
    idx = rng.choice(W * H, size=n_pixels, replace=False)
    ph, pw = (idx // W).astype(np.int32), (idx % W).astype(np.int32)
    fid_all = hash_faceids(seed, W, H, scene.faces_per_light)
    fid = fid_all[idx]
    fs = FlatScene(scene.geom_tri_offset, scene.tri_verts, scene.tri_normals, scene.geom_has_normals,
                   scene.geom_material, scene.light_geom)  # the reference has no spheres
    L = scene.n_lights
    rst = Restated()
    cam12 = rst.camera(EYE, LOOK, W, H)
    strict = None
    if ref_available():
        # headline: the reference's own Release flags (-O3 -ffast-math, cmake/config.cmake:29 -> cmake/gcc.cmake:16);
        # the strict build (the parity oracle) is timed beside it on the same pixels
        def timed(release):
            ref = RefOracle(release=release)
            h = ref.from_flat(fs)
            out = ref.render_pixels(h, W, H, EYE, LOOK, pw, ph, fid, n_threads=threads)
            rays = n_pixels + int((out["geom"] >= 0).sum()) * L
            return ref, h, out["seconds"], rays

        rel = ref_release_available()
        for r_ in ({False, rel}):  # warm both builds (page-in, thread start) on a few pixels before anything is timed
            w_ = RefOracle(release=r_)
            hw_ = w_.from_flat(fs)
            w_.render_pixels(hw_, W, H, EYE, LOOK, pw[:threads], ph[:threads], fid[:threads], n_threads=threads)
            w_.free(hw_)
        ref, h, secs, rays = timed(rel)
        kind, build = "reference", ("-O3 -ffast-math (the reference's Release flags)" if rel else "-O3 -ffp-contract=off (strict)")
        if rel:
            ref.free(h)
            ref_s, h_s, secs_s, rays_s = timed(False)
            strict = dict(value=rays_s / secs_s / 1e6, unit="Mrays/s", seconds=secs_s, build="-O3 -ffp-contract=off (parity oracle)")
            ref.lib, h = ref_s.lib, h_s  # the extras below run on the strict build's handle
            ref = ref_s
    else:
        ref, h = None, None
        t0 = time.time()
        o = rst.render_pixels(fs, cam12, W, H, pw, ph, fid, n_threads=threads)
        secs, kind, build = time.time() - t0, "port", "oracle/restated.c -O2 -ffp-contract=off"
        rays = n_pixels + int((o.tri >= 0).sum()) * L
    out = dict(value=rays / secs / 1e6, unit="Mrays/s", cores=threads, kind=kind, seconds=secs, build=build, strict_build=strict,
               ispc="n/a (no ispc toolchain in this image: src/ispc/trace.ispc cannot be built; it is also semantically "
                    "different and broken upstream, SURVEY App. B)",
               sample=f"{n_pixels} random pixels of the {W}x{H} frame (all {scene.n_tris} triangles, {L} lights; spheres omitted: "
                      f"the reference has none), {'reference intersect()/occlusion() via oracle/_ref' if kind == 'reference' else 'oracle/restated.c'}, "
                      f"{threads} threads")
    if extras and ref is not None:
        # BASELINE.md 3's comparator set: serial on one core, and the reference's --thread scheme (one std::thread per
        # image row sharing one RNG, src/main.cpp:629-643) through the harness' ref_time_rows
        n1 = max(4, n_pixels // max(1, threads) // 2)
        o1 = ref.render_pixels(h, W, H, EYE, LOOK, pw[:n1], ph[:n1], fid[:n1], n_threads=1)
        out["serial_1core"] = dict(value=(n1 + int((o1["geom"] >= 0).sum()) * L) / o1["seconds"] / 1e6, unit="Mrays/s", cores=1,
                                   seconds=o1["seconds"], sample=f"first {n1} pixels of the same sample, 1 thread (strict build)")
        per_px = max(1e-9, secs * threads / n_pixels)                    # core-seconds per pixel, measured above
        Wt = int(max(8, min(W, 6.0 / per_px)))                           # rows of Wt pixels: ~6 s per row thread
        rows = max(1, min(threads, H))
        h0 = (H - rows) // 2
        t_rows = ref.time_rows(h, Wt, H, EYE, LOOK, seed, h0, h0 + rows, 1)
        # every pixel of a closed scene hits, so rays = pixels * (1 + L) to within the miss fraction measured above
        hit_frac = (rays - n_pixels) / max(1, n_pixels * L)
        out["thread_per_row"] = dict(value=rows * Wt * (1 + L * hit_frac) / t_rows / 1e6, unit="Mrays/s", cores=min(rows, threads),
                                     seconds=t_rows, sample=f"{rows} image rows [{h0},{h0 + rows}) of a {Wt}x{H} frame (horizontally "
                                     f"sub-sampled: a full {W}-pixel row is minutes of CPU), one std::thread per row, shared RNG; rays "
                                     f"estimated with the sample's hit fraction {hit_frac:.3f}")
    if ref is not None:
        ref.free(h)
    # SURVEY 8f-4: the same algorithm as a SIMD CPU comparator (oracle/restated.c, 8 triangles per AVX2 step, pinned
    # bit-identical to the scalar restatement), timed on the same pixels: what a vectorised CPU build would reach
    try:
        if rst.set_simd(True):
            t0 = time.time()
            o = rst.render_pixels(fs, cam12, W, H, pw, ph, fid, n_threads=threads)
            dt = time.time() - t0
            out["simd_comparator"] = dict(value=(n_pixels + int((o.tri >= 0).sum()) * L) / dt / 1e6, unit="Mrays/s", cores=threads,
                                          kind="port", seconds=dt, simd="AVX2, 8 triangles per step", sample="same pixels as cpu_baseline")
        rst.set_simd(False)
    except Exception as e:  # the comparator is optional
        out["simd_comparator"] = {"unavailable": str(e)[:200]}
    return out


def sample_size(scene, W, H, threads, seconds):
    per_px = scene.n_tris * 3.0 / 55e6  # ~55 M tests/s/core (SURVEY 6)
    return int(max(threads, min(W * H, seconds * threads / max(per_px, 1e-6))))


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation on the host cores, same metric/config."""
    if rank != 0:
        return
    scene, W, H = make_scene(args.workload, args)
    spp = args.spp or WORKLOAD_SPP.get(args.workload, 0)
    threads = os.cpu_count() or 1
    n_px = sample_size(scene, W, H, threads, 20.0 / max(1, args.steps + args.warmup))
    for _ in range(args.warmup):
        cpu_sample(scene, W, H, max(threads, n_px // 4), threads)
    vals, secs = [], 0.0
    for _ in range(args.steps):
        c = cpu_sample(scene, W, H, n_px, threads)
        vals.append(c["value"])
        secs += c["seconds"]
    v = float(np.mean(vals))
    c["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": "Mrays/s (primary+shadow)", "value": v, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, scene, W, H, spp, args.mode), "cpu_baseline": c,
        "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "libtracer_cuda_loaded": any("libtracer_cuda" in l for l in open("/proc/self/maps")),
    }))


def pinned_scene(scene):
    """the same scene with every array in page-locked host memory (what a host flow that feeds a GPU would hold)"""
    import torch

    from esctp1raytracer_b200 import Scene

    keep = []

    def pin(a):
        if a is None:
            return None
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()

    sc = Scene(pin(scene.geom_tri_offset), pin(scene.tri_verts), pin(scene.geom_material), pin(scene.light_geom),
               tri_normals=pin(scene.tri_normals), geom_has_normals=pin(scene.geom_has_normals),
               sphere_cr=pin(scene.sphere_cr), sphere_material=pin(scene.sphere_material))
    sc._pinned = keep
    return sc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--tris", type=int, default=0)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cull", action="store_true", help="skip the extra measurement of the optional bundle-cull mode")
    ap.add_argument("--mode", default="brute", choices=["brute", "cull"],
                    help="which mode `value` measures; the default is the north star's brute-force formulation")
    ap.add_argument("--spp", type=int, default=0, help="samples per pixel (extension); default: the workload's")
    ap.add_argument("--native-dist", action="store_true",
                    help="ONE process drives --gpus N GPUs through the library's own multi-GPU entry points (NCCL inside the C ABI) "
                         "instead of one rank per GPU under torchrun")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the frame the last timed step rendered to DIR/*.npy (float32), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU frame; --impl reference times a pixel sample and renders no frame")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    from esctp1raytracer_b200 import Camera, MultiRenderer, Renderer
    from esctp1raytracer_b200 import dist as tdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    native = args.native_dist and world == 1 and args.gpus > 1
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    scene, W, H = make_scene(args.workload, args)
    cam = Camera.for_frame(EYE, LOOK, W, H)
    seed = 42
    spp = args.spp or WORKLOAD_SPP.get(args.workload, 0)
    main_cull = args.mode == "cull"
    n_gpus = args.gpus if native else world

    if native:
        multi = MultiRenderer(args.gpus)
        renderer = Renderer.__new__(Renderer)  # peak / device info only: same library, GPU 0 is the current context
        renderer.lib, renderer.device = multi.lib, 0
        host_out = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()

        def upload(sc):
            return multi.upload(sc)

        dev_frame = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda:0")

        def render(rs, cull):  # like the torch path, `value` leaves the assembled frame in HBM on GPU 0
            fr = multi.trace(rs, cam, W, H, seed=seed, bundle_cull=cull, samples_per_pixel=spp, out_device_ptr=dev_frame.data_ptr())
            return dev_frame, fr.stats
    else:
        renderer = Renderer(local_rank)

        def upload(sc):
            return renderer.upload(sc)

        def render(rs, cull):
            return tdist.render_frame(renderer, rs, cam, W, H, rank=rank, world=world, seed=seed, bundle_cull=cull,
                                      samples_per_pixel=spp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- FP32 peak of this GPU, measured now ----------------------------------------------
    # variants 0/3 scalar FFMA chains, 1 packed FFMA2 chains.  (Variant 2, an instruction-mix kernel, is not a
    # peak: the compiler hoists part of its FFMAs, so its flop count over-states what was executed.)
    peaks = {v: renderer.fp32_peak(v, 5)[0] for v in (0, 1, 3)}
    peak_tflops = max(peaks.values())
    info = renderer.device_info()
    nominal = info["sm_count"] * 128 * 2 * info["clock_khz"] * 1e3 / 1e12

    # ---- value: resident scene, frame stays in HBM ------------------------------------------
    rs = upload(scene)
    # nvidia-smi is started BEFORE the warm-up: its start-up (NVML initialisation, a few hundred ms during which driver
    # calls can stall) must not fall into the timed region; only the samples taken inside the region are reported
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        render(rs, main_cull)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    acc = {}
    barrier()
    sampler.mark()
    t_wall = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        frame, st = render(rs, main_cull)
        for k, v in st.items():
            acc[k] = acc.get(k, 0) + v
    ev1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    # native: the frames are produced on the library's own streams by its host threads; torch's events on this thread's
    # stream do not bracket them, the wall clock around the (blocking) calls does
    ms = t_wall * 1e3 if native else ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    frame_sha = hashlib.sha256(frame.cpu().numpy().tobytes()).hexdigest() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, frame.cpu().numpy())
    flop_primary = float(st.get("flop_primary") or 0.0)  # FP32 flops executed per swept pair (same on every rank)
    flop_shadow = float(st.get("flop_shadow") or 0.0)
    flop_primary_e = float(st.get("flop_primary_edges") or 0.0)
    flop_shadow_e = float(st.get("flop_shadow_edges") or 0.0)
    keys = ["n_primary_rays", "n_shadow_rays", "tests_primary", "tests_shadow", "tests_shadow_ref", "strict_evals",
            "kernel_launches", "ms_primary", "ms_shadow", "ms_total"]
    t = torch.tensor([ms] + [float(acc.get(k, 0)) for k in keys], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms = float(mx[0])
        sweep_ms_max = float(mx[8] + mx[9])
    else:
        sweep_ms_max = float(t[8] + t[9])  # native: the library already reports the slowest GPU's times
    tot = {k: float(t[i + 1]) for i, k in enumerate(keys)}
    rays = tot["n_primary_rays"] + tot["n_shadow_rays"]
    value = rays / (ms * 1e-3) / 1e6
    launches = int(tot["kernel_launches"]) + (args.steps if world > 1 else 0)

    # ---- extra: the OPTIONAL bundle-cull mode (same frame, hierarchical evaluation of the same filter) ------
    cull_extra = None
    if not args.no_cull and not main_cull:
        for _ in range(2):
            frame_c, _ = render(rs, True)
        same = bool(torch.equal(frame.cpu(), frame_c.cpu())) if rank == 0 else True
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tc = time.perf_counter()
        c0.record()
        for _ in range(args.steps):
            render(rs, True)
        c1.record()
        barrier()
        tc = time.perf_counter() - tc
        cms = torch.tensor([tc * 1e3 if native else c0.elapsed_time(c1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(cms, op=dist.ReduceOp.MAX)
        cull_extra = {"value": rays / (float(cms[0]) * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": float(cms[0]) / args.steps,
                      "frame_identical_to_default_mode": same,
                      "frame_sha256": hashlib.sha256(frame_c.cpu().numpy().tobytes()).hexdigest() if rank == 0 else None,
                      "note": "opts.bundle_cull (two-phase): every (ray block, triangle) pair against the block box, survivors against "
                              "the 16 warp boxes -> sorted per-(block, warp) lists -> lane box -> per-ray filter -> strict pairs merged "
                              "by atomicMin; no acceleration structure, results bit-identical.  "
                              "Reported beside the headline, which stays on the brute-force per-ray formulation of the north star."}

    # ---- e2e: host buffers in, host frame out, every step --------------------------------------------
    e2e = None
    if not args.no_e2e:
        h2d = int(scene.tri_verts.nbytes + (scene.tri_normals.nbytes if scene.tri_normals is not None else 0)
                  + scene.geom_material.nbytes + scene.n_tris * 4 + scene.sphere_cr.nbytes
                  + scene.sphere_material.nbytes + 48)
        pin = pinned_scene(scene)
        host_frame = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() if rank == 0 else None
        if world == 1 and not native:
            # the literal drop-in call: tracer_cuda_render(scene, camera, W, H, opts, rgb_out), host pointers both ways
            def e2e_step():
                renderer.trace(pin, cam, W, H, seed=seed, bundle_cull=main_cull, samples_per_pixel=spp, out=host_frame.numpy())
            path = "tracer_cuda_render(host scene, camera, W, H, opts, host rgb_out): upload + table build + render + read-back in one C call"
        elif native:
            def e2e_step():
                fr = multi.trace(pin, cam, W, H, seed=seed, bundle_cull=main_cull, samples_per_pixel=spp)
                host_frame.numpy()[...] = fr.rgb8  # (MultiRenderer returns its own host array)
            path = "tracer_cuda_render_multi(host scene, ...): per-GPU upload + render + NCCL gather + read-back in one C call"
        else:
            def e2e_step():
                r2 = renderer.upload(pin)  # host -> HBM every step, on every rank
                fr, _ = render(r2, main_cull)
                if rank == 0:
                    host_frame.copy_(fr, non_blocking=False)  # HBM -> host read of the result
                r2.close()
            path = "per rank: tracer_cuda_scene_create(host scene) + band render + NCCL gather; rank 0 reads the assembled frame back"

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_sha = hashlib.sha256(host_frame.numpy().tobytes()).hexdigest() if rank == 0 else None
        e2e = {"value": rays / float(dt[0]) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": h2d * n_gpus,
               "d2h_bytes_per_step": W * H * 3, "ms_per_step": float(dt[0]) / args.steps * 1e3, "path": path,
               "host_memory": "pinned (scene arrays and the frame)", "frame_sha256": e2e_sha,
               "includes": "scene upload + filter-table build + render + band gather + frame read-back"}

    if rank == 0:
        alg_pairs = tot["tests_primary"] + tot["tests_shadow_ref"]
        swept_pairs = tot["tests_primary"] + tot["tests_shadow"]
        sweep_s = max(sweep_ms_max * 1e-3, 1e-12)
        alg_flop = flop_primary * tot["tests_primary"] + flop_shadow * tot["tests_shadow_ref"]
        # FMA-pipe view: every FADD / FMUL / FFMA is one lane-operation of the pipe whose peak is peak_tflops / 2 lane-ops
        # per second (an FFMA counts two flops, a saturating FADD one, yet both hold a lane for one cycle); a packed FFMA2
        # is two.  Span form: 2 FADD.SAT + half an FFMA2 per pair + the bound FFMAs per thread = 3 + (flop - 4) / 2;
        # three-row form with own q (jittered samples): 6 FFMA.SAT + FMUL + FFMA = 8
        def lane_ops(flop):
            return 8.0 if flop >= 15.0 else (3.0 + (flop - 4.0) / 2.0 if flop > 0 else 0.0)
        alg_lane_ops = lane_ops(flop_primary) * tot["tests_primary"] + lane_ops(flop_shadow) * tot["tests_shadow_ref"]
        swept_flop = flop_primary * tot["tests_primary"] + flop_shadow * tot["tests_shadow"]
        achieved = alg_flop / n_gpus / sweep_s / 1e12  # per GPU
        achieved_lane = alg_lane_ops / n_gpus / sweep_s / 1e12  # T lane-ops/s per GPU
        # As issued: ptxas folds the exact power-of-two scaling of p into each saturating add (FFMA.SAT R, p, 65536, ax,
        # profiles/r02_l_sass_primary_span_hot_loop.txt), so the SASS executes two FFMA where the formulation needs two
        # FADD: +2 flops per pair on the span form.  Reported beside the fraction, never as it.
        def issued(flop):
            return flop if flop >= 15.0 or flop <= 0 else flop + 2.0
        issued_flop = issued(flop_primary) * tot["tests_primary"] + issued(flop_shadow) * tot["tests_shadow_ref"]
        achieved_issued = issued_flop / n_gpus / sweep_s / 1e12
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            pass
        prim_bytes = 32.0 * scene.n_tris * (1 + scene.n_lights * 2) + 36.0 * scene.n_tris
        hbm_gbs = (prim_bytes + 3.0 * W * H / n_gpus) * args.steps / (ms * 1e-3) / 1e9
        traffic = traffic_detail = None  # dram bytes per launch of the dominant kernel, from the committed ncu --set full capture
        for tf in ("r02_traffic.json", "r01_traffic.json"):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", tf)))
                traffic = tj["traffic_bytes_per_launch"]
                traffic_detail = {"algorithmic_bytes_per_launch": tj["algorithmic_bytes_per_launch"], "kernel": tj["kernel"],
                                  "capture_config": tj["config_of_capture"], "source": tj["capture"], "note": tj.get("algorithmic_note")}
                break
            except Exception:
                pass
        cpu = None
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            cpu = cpu_sample(scene, W, H, sample_size(scene, W, H, threads, 12.0), threads, extras=True)
        ms_prim = tot["ms_primary"] / (1 if native else n_gpus)
        ms_shad = tot["ms_shadow"] / (1 if native else n_gpus)
        prim_tflops = flop_primary * tot["tests_primary"] / n_gpus / (ms_prim * 1e-3) / 1e12 if ms_prim else None
        line = {
            "metric": "Mrays/s (primary+shadow)", "value": value, "unit": "Mrays/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, scene, W, H, spp, args.mode),
            "multi_gpu_path": ("one process, tracer_cuda_init_multi: host thread per GPU, grouped ncclSend/ncclRecv inside the C ABI" if native
                               else "one process per GPU (torchrun), torch.distributed NCCL gather of the packed bands" if world > 1 else "single GPU"),
            "frame_sha256": frame_sha,
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "roofline": {
                "bound": "fp32", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s", "frac": achieved / peak_tflops,
                "traffic": traffic, "traffic_detail": traffic_detail,
                "peak_source": "own FFMA/FFMA2 microbenchmark in this process (tracer_cuda_fp32_peak): best of scalar FFMA chains "
                               "(variants 0, 3) and packed FFMA2 chains (variant 1); MEASURED_PEAKS.json has no FP32 figure",
                "peak_nominal": nominal, "frac_of_nominal": achieved / nominal, "peak_variants_tflops": peaks,
                "peak_scalar_ffma": max(peaks[0], peaks[3]), "frac_of_scalar_ffma_peak": achieved / max(peaks[0], peaks[3]),
                "flop_per_pair": {"primary": flop_primary, "shadow": flop_shadow, "primary_bounds_only": flop_primary_e,
                                  "shadow_bounds_only": flop_shadow_e,
                                  "note": "FP32 flops the sweeps execute per (ray, triangle) pair, all in the FMA pipe (FFMA = 2, FADD = 1).  "
                                          "Span form (csrc/sweep.cuh): for rays that share q the three affine edge rows of a triangle are "
                                          "two lower and two upper bounds of p; per thread and triangle 4 FFMA + 2 FMNMX evaluate them "
                                          "(closest hit: R = 32 pixels of one image row share q exactly; shadow: 8 FFMA, R = 16 q-sorted rays "
                                          "share mean q + |B| * spread, still a necessary condition); per PAIR x = sat(S p + ax), "
                                          "y = sat(ay - S p) (2 FADD.SAT = 2 flops) and acc += x*y (half a packed FFMA2 = 2 flops): "
                                          "4 + 8/R resp. 4 + 16/R flops.  No integer/ALU-pipe instruction per pair.  Because half of the "
                                          "per-pair instructions are adds (1 flop per lane-cycle instead of 2) the flop fraction under-states "
                                          "how busy the FMA pipe is: see fma_pipe"},
                "mix_ceiling_frac": alg_flop / (2.0 * alg_lane_ops) if alg_lane_ops else None,
                "mix_ceiling_note": "the fraction this instruction mix would reach with every FMA-pipe lane-cycle used: saturating adds "
                                    "count 1 flop per lane-cycle, multiply-adds 2 (SURVEY 8d asks for this ceiling beside every fraction)",
                "as_issued": {"flop_per_pair": {"primary": issued(flop_primary), "shadow": issued(flop_shadow)},
                              "tflops": achieved_issued, "frac": achieved_issued / peak_tflops, "frac_of_nominal": achieved_issued / nominal,
                              "note": "NOT roofline.frac: the SASS issues each saturating add as FFMA.SAT with an immediate scale "
                                      "(R = sat(p * 65536 + ax); the product is exact), i.e. the FMA pipe executes 6 + 8/R flops per pair; "
                                      "roofline.frac counts the 4 + 8/R the formulation needs"},
                "fma_pipe": {"lane_ops_per_pair": {"primary": lane_ops(flop_primary), "shadow": lane_ops(flop_shadow)},
                             "achieved_tlaneops": achieved_lane, "peak_tlaneops": peak_tflops / 2.0, "frac": achieved_lane / (peak_tflops / 2.0),
                             "frac_of_nominal": achieved_lane / (nominal / 2.0),
                             "note": "FMA-pipe lane-operations (FADD, FMUL, FFMA = 1 each, packed FFMA2 = 2) of the algorithmic pairs per "
                                     "second against the measured peak in the same unit (peak TFLOP/s / 2): the issue-slot view of the "
                                     "same kernel time"},
                "algorithmic_pairs_per_step": alg_pairs / args.steps,
                "swept_pairs_per_step": swept_pairs / args.steps, "sweep_ms_per_step": sweep_ms_max / args.steps,
                "executed_tflops": swept_flop / n_gpus / sweep_s / 1e12,
                "primary_ms_per_step": ms_prim / args.steps, "shadow_ms_per_step": ms_shad / args.steps,
                "primary_tflops": prim_tflops,
                "dominant_kernel": {
                    "kernel": "trk::primary_kernel (closest-hit sweep, one launch per frame)",
                    "achieved": prim_tflops, "unit": "TFLOP/s", "frac": prim_tflops / peak_tflops if prim_tflops else None,
                    "frac_of_nominal": prim_tflops / nominal if prim_tflops else None,
                    "share_of_sweep_time": ms_prim / (ms_prim + ms_shad) if (ms_prim + ms_shad) else None,
                    "note": "the launch the roofline contract names (algorithmic flops of that launch / its duration, CUDA events "
                            "inside the library).  roofline.frac above is the more conservative figure over BOTH sweeps (this "
                            "launch + the per-light shadow launches, shadow pairs at the reference's own in-order count)"},
                "shadow_tflops": flop_shadow * tot["tests_shadow"] / n_gpus / (ms_shad * 1e-3) / 1e12 if ms_shad else None,
                "pair_rate_tpairs_s": swept_pairs / n_gpus / sweep_s / 1e12,
                "reference_formulation_tflops": FLOP_PER_PAIR_REF * alg_pairs / n_gpus / sweep_s / 1e12,
                "ceiling_note": "the loop is FMA-pipe issue bound: on this part a scalar FMA-pipe instruction costs ~1.3 issue cycles (own "
                                "microbenchmark: scalar FFMA chains peak at 0.745 per cycle and scheduler = peak_scalar_ffma; only packed FFMA2 "
                                "reaches 0.92), independent of occupancy; per pair the loop issues 2 FADD.SAT + FFMA2/2, per thread and "
                                "triangle 4 (shadow: 8) FFMA + 2 FMNMX + 2 LDS.128 (tools/sweep_mb4.cu: 9.5 Tpairs/s at R = 32, "
                                "8.2 at R = 16 with shared mean q; profiles/r02_*)",
                "hbm": {"achieved_gbs": hbm_gbs, "peak_gbs": hbm_peak, "frac": (hbm_gbs / hbm_peak) if hbm_peak else None,
                        "streams": "span tables (32 B/triangle/origin) + vertices (36 B/triangle) + framebuffer (3 B/pixel)"},
            },
            "cpu_baseline": cpu, "optional_bundle_cull_mode": cull_extra,
            "rays_per_step": rays / args.steps, "strict_evals_per_step": tot["strict_evals"] / args.steps,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
