"""The seeded std::mt19937 mode (RNG_MT19937) replayed on the device, in row bands and on several GPUs.

* the device replay (tracer__mt19937_faceids_device) against tracer_mt19937_faceids at full size: a 3840x2160 mask with
  4 lights of 2 faces, and a 10^6-pixel mask with face counts that reject 25-30 % of draws;
* bands on one GPU: every band of (2, 8), (3, 5), (4, 8) and (8, 16) (band_rows, band_count) of the golden frames and the
  full-size C1/C3 frames, with an exchange hook that checks its own rows and fills the rest from a whole-frame render,
  assembles to the reference's PPM bytes, with the whole-frame render's debug outputs; also in bundle-cull and BVH modes;
* a bundle-cull closest-hit pass that overflows its candidate buffer: rendered again before its row counts are used;
* misuse: a failing hook, a hook that alters its own rows, bands without a hook;
* several GPUs (skipped with one): MultiRenderer, tracer_cli --gpus, dist.render_frame under torch.multiprocessing.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import GOLDEN, ROOT, golden_names, load_golden, to_scene
from test_mt19937_replay import REJECTING, reference_faceids

pytestmark = pytest.mark.gpu

BANDS = [(2, 8), (3, 5), (4, 8), (8, 16)]


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


def _n_gpus():
    import torch

    return torch.cuda.device_count()


def device_faceids(renderer, faces, W, H, seed, hit_img):
    lib = renderer.lib
    lib.tracer__mt19937_faceids_device.argtypes = [C.c_uint32, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_int32,
                                                   C.POINTER(C.c_uint8), C.POINTER(C.c_int32), C.POINTER(C.c_double)]
    L = len(faces)
    f = np.asarray(faces, np.int32)
    scan = np.ascontiguousarray(np.asarray(hit_img, np.uint8).reshape(H, W)[::-1]).reshape(-1)
    out = np.full((W * H, L), -7, np.int32)
    ms = C.c_double()
    from esctp1raytracer_b200 import _lib

    _lib.check(lib.tracer__mt19937_faceids_device(seed, L, f.ctypes.data_as(C.POINTER(C.c_int32)), W, H,
                                                  scan.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                  out.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(ms)))
    return out.reshape(H, W, L)[::-1].reshape(W * H, L)


def test_device_faceids_at_full_size(renderer):
    from esctp1raytracer_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(4)
    W, H = 3840, 2160
    hit = rng.random(W * H) < 0.9
    assert np.array_equal(device_faceids(renderer, [2] * 4, W, H, 42, hit), reference_faceids(lib, [2] * 4, W, H, 42, hit))
    W, H = 1000, 1000
    faces = [REJECTING[0], REJECTING[1], 7]
    hit = rng.random(W * H) < 0.7
    assert np.array_equal(device_faceids(renderer, faces, W, H, 9, hit), reference_faceids(lib, faces, W, H, 9, hit))


def _frames():
    from test_gpu_fullsize import _load_full

    for name in golden_names():
        fs, fr = load_golden(name)
        yield name, to_scene(fs), fr["eye"], fr["look"], fr["W"], fr["H"], fr["seed"], fr["q"]
    for name in ("c1_cornell_original_1024x768", "c3_sphere_1080p", "c3_water_1080p"):
        if os.path.exists(os.path.join(GOLDEN, "full", name + ".npz")):
            sc, z = _load_full(name)
            yield name, sc, z["eye"], z["look"], int(z["W"]), int(z["H"]), int(z["seed"]), z["q"]


def _checking_hook(frame_rows, own):
    """the exchange: this call's rows arrive as the whole-frame render counts them, 0 elsewhere; fills in the rest"""
    calls = []

    def hook(row_hits):
        want = np.where(own, frame_rows, 0)
        assert np.array_equal(row_hits, want), "row counts on entry"
        row_hits[:] = frame_rows
        calls.append(1)

    return hook, calls


@pytest.mark.parametrize("mode", ["sweeps", "bundle_cull", "bvh"])
def test_bands_on_one_gpu_equal_the_seeded_frame(renderer, mode):
    from esctp1raytracer_b200 import RNG_MT19937, Camera

    kw = dict(bundle_cull=mode == "bundle_cull", bvh=mode == "bvh")
    for name, sc, eye, look, W, H, seed, q in _frames():
        cam = Camera.for_frame(eye, look, W, H)
        rs = renderer.upload(sc)
        whole = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=seed, debug=True, **kw)
        assert np.array_equal(whole.rgb8.reshape(-1, 3), np.asarray(q, np.uint8).reshape(-1, 3)), name
        frame_rows = (whole.tri.reshape(H, W) >= 0).sum(1).astype(np.int32)  # PPM row order
        for band_rows, n in BANDS:
            rgb8 = np.zeros_like(whole.rgb8)
            dbg = {k: np.zeros_like(getattr(whole, k).reshape(H, W, -1)) for k in ("tri", "t", "v", "occ_tri", "rgb")}
            for bi in range(n):
                rows = [pr for pr in range(H) if (pr // band_rows) % n == bi]
                own = np.zeros(H, bool)
                own[rows] = True
                hook, calls = _checking_hook(frame_rows, own)
                part = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=seed, bands=(band_rows, bi, n), debug=True,
                                      row_hits_exchange=hook, **kw)
                assert len(calls) == 1, (name, band_rows, n, bi)
                rgb8[rows] = part.rgb8
                for k in dbg:
                    dbg[k][rows] = getattr(part, k).reshape(len(rows), *dbg[k].shape[1:])
            assert np.array_equal(rgb8, whole.rgb8), (name, band_rows, n)
            for k, a in dbg.items():  # bit for bit
                assert a.tobytes() == getattr(whole, k).reshape(H, W, -1).tobytes(), (name, band_rows, n, k)
        rs.close()


def test_bundle_cull_overflow_gives_the_seeded_frame(renderer, monkeypatch):
    """A bundle-cull closest-hit pass whose candidates overflow has lost hits: the frame is rendered again before any row
    count is used or exchanged (TRACER_CAND_CAP fakes a tiny candidate buffer), whole frames and hooked bands alike."""
    from esctp1raytracer_b200 import RNG_MT19937, Camera, scenes

    s = scenes.soup_scene(20000, 40, 3, seed=6)
    W, H = 96, 64
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    want = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, debug=True)
    frame_rows = (want.tri.reshape(H, W) >= 0).sum(1).astype(np.int32)
    monkeypatch.setenv("TRACER_CAND_CAP", "1000")
    for mode in (1, 2):
        got = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, debug=True, bundle_cull=mode)
        assert got.stats["flop_primary"] > 0  # rendered again by the default sweeps
        for k in ("rgb8", "tri", "occ_tri", "rgb"):
            assert getattr(got, k).tobytes() == getattr(want, k).tobytes(), (mode, k)
        rgb8 = np.zeros_like(want.rgb8)
        for bi in range(3):
            rows = [pr for pr in range(H) if (pr // 8) % 3 == bi]
            own = np.zeros(H, bool)
            own[rows] = True
            hook, calls = _checking_hook(frame_rows, own)
            part = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, bands=(8, bi, 3), bundle_cull=mode,
                                  row_hits_exchange=hook)
            assert len(calls) == 1
            rgb8[rows] = part.rgb8
        assert np.array_equal(rgb8, want.rgb8), mode


def test_misuse(renderer):
    from esctp1raytracer_b200 import RNG_MT19937, Camera, TracerError, scenes

    s = scenes.box_scene()
    W, H = 100, 77
    cam = Camera.for_frame((0, 1, 2.9), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    whole = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, debug=True)
    frame_rows = (whole.tri.reshape(H, W) >= 0).sum(1).astype(np.int32)

    def broken(row_hits):
        raise RuntimeError("the exchange failed")

    with pytest.raises(TracerError, match="error -5"):
        renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, bands=(8, 1, 2), row_hits_exchange=broken)
    again = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, debug=True)
    assert np.array_equal(again.rgb8, whole.rgb8) and np.array_equal(again.tri, whole.tri)

    def alters_own(row_hits):
        row_hits[:] = frame_rows
        row_hits[8] += 1  # PPM row 8 belongs to band 1 of (8, 2)

    with pytest.raises(TracerError, match="error -1"):
        renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, bands=(8, 1, 2), row_hits_exchange=alters_own)

    def out_of_range(row_hits):
        row_hits[:] = frame_rows
        row_hits[0] = W + 1  # not this call's row, but no row has more than W hits

    with pytest.raises(TracerError, match="error -1"):
        renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, bands=(8, 1, 2), row_hits_exchange=out_of_range)
    with pytest.raises(TracerError, match="row_hits_exchange"):
        renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, bands=(8, 1, 2))
    # a band selection with no rows still takes part in the exchange
    hook, calls = _checking_hook(frame_rows, np.zeros(H, bool))
    part = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3, bands=(64, 3, 4), row_hits_exchange=hook)
    assert len(calls) == 1 and part.rgb8.shape[0] == 0
    assert np.array_equal(renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=3).rgb8, whole.rgb8)


def test_multi_gpu_seeded_frames_equal_one_gpu():
    from esctp1raytracer_b200 import RNG_MT19937, Camera, MultiRenderer, Renderer, scenes

    n = _n_gpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    s = scenes.soup_scene(30000, 30, 3, seed=9, n_spheres=5)
    W, H = 200, 121
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    one = Renderer(0)
    want = one.trace(one.upload(s), cam, W, H, rng_mode=RNG_MT19937, seed=4).rgb8
    for k in sorted({2, n}):
        m = MultiRenderer(k)
        rs = m.upload(s)
        assert np.array_equal(m.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=4).rgb8, want), f"{k}-GPU frame differs"
        assert np.array_equal(m.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=4, band_rows=5).rgb8, want)
        assert np.array_equal(m.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=4, bundle_cull=True).rgb8, want)
        rs.close()
        assert np.array_equal(m.trace(s, cam, W, H, rng_mode=RNG_MT19937, seed=4).rgb8, want)  # the drop-in call


def test_cli_gpus_seeded_writes_the_one_gpu_ppm(tmp_path):
    from conftest import write_obj

    from esctp1raytracer_b200 import scenes

    n = _n_gpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    obj = tmp_path / "box.obj"
    write_obj(scenes.box_scene(), obj)
    cli = os.path.join(ROOT, "esctp1raytracer_b200", "tracer_cli.bin")
    outs = []
    for k in (1, n):
        out = tmp_path / f"out{k}.ppm"
        r = subprocess.run([cli, "-m", str(obj), "-v", "0,1,2.9", "-l", "0,1,0", "-w", "160,100", "--seed", "5",
                            "--gpus", str(k), "-o", str(out)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(out.read_bytes())
    assert outs[0] == outs[1]


def _rank_main(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    from esctp1raytracer_b200 import RNG_MT19937, Camera, Renderer, scenes
    from esctp1raytracer_b200 import dist as tdist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    r = Renderer(rank)
    s = scenes.soup_scene(30000, 30, 3, seed=9, n_spheres=5)
    W, H = 200, 121
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = r.upload(s)
    frame, _ = tdist.render_frame(r, rs, cam, W, H, rank=rank, world=world, rng_mode=RNG_MT19937, seed=4)
    if rank == 0:
        want = r.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=4).rgb8
        q.put(bool(np.array_equal(frame.cpu().numpy(), want)))
    dist.destroy_process_group()


def test_torch_distributed_seeded_frame_equals_single_gpu():
    import torch.multiprocessing as mp

    n = _n_gpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29900 + os.getpid() % 400
    procs = [ctx.Process(target=_rank_main, args=(r, n, port, q)) for r in range(n)]
    for p in procs:
        p.start()
    ok = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
    assert ok is True
