"""The optional BVH mode (opts.accel = 1, csrc/bvh.cuh) on the GPU: the reference's own frames, and bit-identical debug
outputs to the default mode on the scenes the bundle-cull mode is held to, with bands, multi-sample and the seeded
mt19937 mode; the full C4 frame; invalid combinations; multi-GPU; the CLI's --bvh."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits, golden_names, load_golden, to_flat, to_scene

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


def _ppm(a, W, H):
    return a.reshape(H, W, *a.shape[1:])[::-1].reshape(a.shape)


def _same_frames(a, b):
    assert np.array_equal(a.rgb8, b.rgb8)
    assert np.array_equal(a.tri, b.tri) and np.array_equal(bits(a.t), bits(b.t)) and np.array_equal(bits(a.v), bits(b.v))
    assert np.array_equal(a.occ_tri, b.occ_tri) and np.array_equal(bits(a.rgb), bits(b.rgb))


def _bvh_stats_consistent(st):
    assert st["tests_primary"] + st["tests_shadow"] == st["strict_evals"]
    assert st["flop_primary"] == 0 and st["flop_shadow"] == 0 and st["filter_misses"] == 0


@pytest.mark.parametrize("name", golden_names())
def test_bvh_golden(renderer, name):
    """the reference's small frames, faceIDs replayed: ids, t, v, float accumulator, PPM bytes"""
    from esctp1raytracer_b200 import Camera, RNG_EXPLICIT

    fs, fr = load_golden(name)
    W, H = fr["W"], fr["H"]
    cam = Camera.for_frame(fr["eye"], fr["look"], W, H)
    out = renderer.trace(renderer.upload(to_scene(fs)), cam, W, H, rng_mode=RNG_EXPLICIT, faceid=fr["faceid"], debug=True, bvh=True)
    assert np.array_equal(out.tri, _ppm(fr["tri"], W, H))
    assert np.array_equal(bits(out.t), bits(_ppm(fr["t"], W, H))) and np.array_equal(bits(out.v), bits(_ppm(fr["v"], W, H)))
    assert np.array_equal(bits(out.rgb), bits(_ppm(fr["rgb"], W, H)))
    assert np.array_equal(out.rgb8.reshape(-1, 3), np.asarray(fr["q"], np.uint8).reshape(-1, 3))
    _bvh_stats_consistent(out.stats)


def test_bvh_full_size_goldens(renderer):
    """C1 and C3 Sphere / Water at their configured sizes (geometry and sorted order): the reference's frames"""
    import test_gpu_fullsize as fsz
    from esctp1raytracer_b200 import Camera, RNG_EXPLICIT

    for name in fsz.FULL:
        sc, z = fsz._load_full(name)
        W, H = int(z["W"]), int(z["H"])
        cam = Camera.for_frame(z["eye"], z["look"], W, H)
        out = renderer.trace(renderer.upload(sc), cam, W, H, rng_mode=RNG_EXPLICIT, faceid=z["faceid"].astype(np.int32), debug=True,
                             bvh=True)
        fsz._check_against_reference(out, z, W, H)


def test_bvh_identical_to_default(renderer):
    from esctp1raytracer_b200 import RNG_HASH, RNG_MT19937, Camera, scenes

    cases = [
        (scenes.soup_scene(20000, 40, 4, seed=5), 96, 64, (0, 1, 3)),
        (scenes.soup_scene(6000, 20, 2, seed=9, edge=(0.05, 0.2), with_normals=True, specular=True, n_spheres=30), 80, 60, (0, 1, 3)),
        (scenes.coplanar_scene(), 120, 90, (0, 1, 2.9)),
        (scenes.soup_scene(60000, 60, 4, seed=1), 333, 187, (0.3, 1.2, 2.7)),
    ]
    for s, W, H, eye in cases:
        cam = Camera.for_frame(eye, (0, 1, 0), W, H)
        rs = renderer.upload(s)
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True)
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bvh=True)
        _same_frames(a, b)
        assert b.stats["tests_shadow_ref"] == a.stats["tests_shadow_ref"] and b.stats["n_shadow_rays"] == a.stats["n_shadow_rays"]
        _bvh_stats_consistent(b.stats)
        c = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bvh=True)  # the kept tree
        _same_frames(a, c)
    # one-shot call (the tree is built inside it), bands assembled into a frame, 2x2 spp, the seeded mt19937 mode
    s, W, H = cases[0][0], 100, 77
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    full = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4).rgb8
    assert np.array_equal(renderer.trace(s, cam, W, H, rng_mode=RNG_HASH, seed=4, bvh=True).rgb8, full)
    frame = np.zeros_like(full)
    for r in range(3):
        part = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, bands=(8, r, 3), bvh=True).rgb8
        frame[[pr for pr in range(H) if (pr // 8) % 3 == r]] = part
    assert np.array_equal(frame, full)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, samples_per_pixel=4)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, samples_per_pixel=4, bvh=True)
    assert np.array_equal(a.rgb8, b.rgb8)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=7, debug=True)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=7, debug=True, bvh=True)
    _same_frames(a, b)


def test_bvh_huge_and_degenerate_triangles(renderer, restated):
    """big triangles all around the eye and lights (always-test list), axis-aligned edges, needles, zero-area triangles,
    triangles through the eye's plane"""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    rng = np.random.default_rng(5)
    s = scenes.soup_scene(200, 6, 2, seed=31, edge=(0.2, 1.5))
    v = s.tri_verts.reshape(-1, 3, 3).copy()
    for i in range(8, 40):
        v[i, 1] = v[i, 0] + np.array([rng.uniform(0.2, 2.0), 0.0, 0.0], np.float32)
        v[i, 2] = v[i, 0] + np.array([0.0, rng.uniform(0.2, 2.0), 0.0], np.float32)
    for i in range(40, 60):
        v[i, 1] = v[i, 0] + np.float32(1e-6) * rng.normal(size=3).astype(np.float32)
        v[i, 2] = v[i, 0] + (v[i, 1] - v[i, 0]) * np.float32(2.0) if i % 2 else v[i, 0]
    for i in range(60, 90):
        v[i, 0, 2], v[i, 1, 2], v[i, 2, 2] = 2.0, 4.5, 3.0
    for i in range(90, 120):  # small ones, in the tree
        v[i] = v[i, 0] + rng.normal(size=(3, 3)).astype(np.float32) * np.float32(0.01)
    s.tri_verts = np.ascontiguousarray(v, np.float32)
    for (W, H, eye, look) in ((160, 90, (0, 1, 3), (0, 1, 0)), (97, 61, (0.3, 0.8, 0.5), (0.1, 1.0, -1.0))):
        cam = Camera.for_frame(eye, look, W, H)
        rs = renderer.upload(s)
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=2, debug=True)
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=2, debug=True, bvh=True)
        _same_frames(a, b)
        o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(2, W, H, s.faces_per_light))
        assert np.array_equal(b.tri, _ppm(o.tri, W, H)) and np.array_equal(b.rgb8.reshape(-1, 3), o.rgb8.reshape(-1, 3))


def test_bvh_invalid_combinations(renderer):
    from esctp1raytracer_b200 import Camera, TracerError, scenes

    s = scenes.soup_scene(1000, 10, 1, seed=2)
    rs = renderer.upload(s)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), 32, 24)
    for kw in (dict(bundle_cull=True), dict(bundle_cull=3), dict(exhaustive_strict=True)):
        with pytest.raises(TracerError, match="-1"):
            renderer.trace(rs, cam, 32, 24, bvh=True, **kw)


def test_bvh_full_size_c4_frame(renderer, restated):
    """the 3840x2160, 1M-triangle + 1k-sphere frame: identical to the default mode, a 96-pixel subset equal to the oracle"""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True, bvh=True)
    _same_frames(a, b)
    _bvh_stats_consistent(b.stats)
    assert b.stats["tests_primary"] < 0.01 * a.stats["tests_primary"]  # the tree prunes
    fid = hash_faceids(seed, W, H, s.faces_per_light)
    idx = np.random.default_rng(1).choice(W * H, 96, replace=False)
    ph, pw = idx // W, idx % W
    o = restated.render_pixels(to_flat(s), cam.as_array(), W, H, pw, ph, fid[idx], n_threads=os.cpu_count() or 1)
    k = (H - 1 - ph) * W + pw
    assert np.array_equal(b.tri[k], o.tri) and np.array_equal(bits(b.t[k]), bits(o.t))
    assert np.array_equal(b.occ_tri[k], o.occ_tri) and np.array_equal(bits(b.rgb[k]), bits(o.rgb))


def test_bvh_multi_gpu_equals_one_gpu(renderer):
    import torch

    from esctp1raytracer_b200 import RNG_HASH, Camera, MultiRenderer, Renderer, scenes

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two or more GPUs")
    s = scenes.soup_scene(20000, 40, 4, seed=5)
    W, H = 200, 150
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    m = MultiRenderer(n)
    got = m.trace(m.upload(s), cam, W, H, rng_mode=RNG_HASH, seed=3, bvh=True).rgb8
    r = Renderer(0)  # back to one GPU
    want = r.trace(r.upload(s), cam, W, H, rng_mode=RNG_HASH, seed=3).rgb8
    assert np.array_equal(got, want)


def test_cli_bvh_equals_sorted(renderer, tmp_path):
    from conftest import write_obj
    from esctp1raytracer_b200 import scenes

    s = scenes.soup_scene(3000, 12, 2, seed=4, edge=(0.03, 0.1))
    obj = tmp_path / "soup.obj"
    write_obj(s, obj)
    cli = os.path.join(ROOT, "esctp1raytracer_b200", "tracer_cli.bin")
    outs = []
    for flag in ("--sorted", "--bvh"):
        out = tmp_path / (flag[2:] + ".ppm")
        r = subprocess.run([cli, "-m", str(obj), "-w", "120,90", "--seed", "17", flag, "-o", str(out)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(out.read_bytes())
    assert outs[0] == outs[1]
    r = subprocess.run([cli, "-m", str(obj), "--thread"], capture_output=True, text=True)
    assert r.returncode != 0
