"""GPU parity: the CUDA path (through the C ABI) against the oracle.

Bar (BASELINE.json north_star): hit ids equal (ties within 1e-5 in t excepted) and PPM
channels within +-1 LSB on >= 99.9 % of pixels.  The strict-finalisation design does
better, and these tests assert it: ids, t, v, occlusion decisions, the float accumulator
and the PPM bytes are BIT-IDENTICAL, specular materials (ks != 0) included, because the
device's powf is glibc's own (strict::powf_glibc, tests/test_powf_glibc.py).
"""
import os

import numpy as np
import pytest
from conftest import bits, golden_names, load_golden, to_flat, to_scene

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


def _cam(fr):
    from esctp1raytracer_b200 import Camera

    return Camera.for_frame(fr["eye"], fr["look"], fr["W"], fr["H"])


def _to_ppm_order(a, W, H):
    """image index order (h*W+w) -> PPM row order (row 0 = h=H-1)"""
    return a.reshape(H, W, *a.shape[1:])[::-1].reshape(a.shape)


def _check_frame(out, W, H, tri, t, v, rgb, q, occ=None):
    assert out.stats == {} or (out.stats["filter_misses"] == 0 and out.stats["pipeline_errors"] == 0)
    assert np.array_equal(out.tri, _to_ppm_order(tri, W, H)), "hit ids differ"
    assert np.array_equal(bits(out.t), bits(_to_ppm_order(t, W, H))), "closest-hit t differs"
    assert np.array_equal(bits(out.v), bits(_to_ppm_order(v, W, H))), "closest-hit v differs"
    if occ is not None:
        assert np.array_equal(out.occ_tri, _to_ppm_order(occ, W, H)), "shadow decisions differ"
    ref_rgb = _to_ppm_order(rgb, W, H)
    assert np.array_equal(bits(out.rgb), bits(ref_rgb)), "float accumulator differs"
    assert np.array_equal(out.rgb8.reshape(-1, 3), np.asarray(q, np.uint8).reshape(-1, 3)), "PPM bytes differ"


@pytest.mark.parametrize("name", golden_names())
def test_golden_explicit_faceids(renderer, name):
    """CUDA vs the frames the reference itself rendered (tests/golden), faceIDs replayed."""
    from esctp1raytracer_b200 import RNG_EXPLICIT

    fs, fr = load_golden(name)
    W, H = fr["W"], fr["H"]
    out = renderer.trace(to_scene(fs), _cam(fr), W, H, rng_mode=RNG_EXPLICIT, faceid=fr["faceid"], debug=True)
    _check_frame(out, W, H, fr["tri"], fr["t"], fr["v"], fr["rgb"], fr["q"])


@pytest.mark.parametrize("name", golden_names())
def test_golden_mt19937_seed(renderer, name):
    """Given only the seed, the library's own std::mt19937 replay reproduces the seeded serial path."""
    from esctp1raytracer_b200 import RNG_MT19937

    fs, fr = load_golden(name)
    W, H = fr["W"], fr["H"]
    rs = renderer.upload(to_scene(fs))
    out = renderer.trace(rs, _cam(fr), W, H, rng_mode=RNG_MT19937, seed=fr["seed"], debug=True)
    _check_frame(out, W, H, fr["tri"], fr["t"], fr["v"], fr["rgb"], fr["q"])
    assert out.stats["kernel_launches"] > 0 and out.stats["tests_primary"] == W * H * fs.n_tris


@pytest.mark.parametrize("name", ["cornell_original", "cornell_sphere", "cornell_original_3lights"])
def test_exhaustive_strict_mode_agrees_and_filter_never_misses(renderer, name):
    from esctp1raytracer_b200 import RNG_EXPLICIT

    fs, fr = load_golden(name)
    W, H = fr["W"], fr["H"]
    rs = renderer.upload(to_scene(fs))
    a = renderer.trace(rs, _cam(fr), W, H, rng_mode=RNG_EXPLICIT, faceid=fr["faceid"], debug=True, exhaustive_strict=True)
    assert a.stats["filter_misses"] == 0 and a.stats["pipeline_errors"] == 0
    _check_frame(a, W, H, fr["tri"], fr["t"], fr["v"], fr["rgb"], fr["q"])


def _soup_case(renderer, restated, n_tris, n_geoms, n_lights, W, H, seed, **kw):
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    s = scenes.soup_scene(n_tris, n_geoms, n_lights, seed=seed, **kw)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    fid = hash_faceids(seed, W, H, s.faces_per_light)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=fid)
    rs = renderer.upload(s)
    out = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True)
    _check_frame(out, W, H, o.tri, o.t, o.v, o.rgb, o.rgb8.reshape(-1, 3), occ=o.occ_tri)
    st = out.stats
    assert st["tests_primary"] == o.n_tests[0]
    assert st["tests_shadow_ref"] == o.n_tests[1]  # the reference's own count of shadow tests
    assert st["n_shadow_rays"] == int((o.tri >= 0).sum()) * n_lights
    return s, rs, cam, out, o


def test_soup_hash_rng_4_lights(renderer, restated):
    """config-4 shaped scene (small): 4 lights, the t carry between lights, counter-based RNG."""
    _soup_case(renderer, restated, 20000, 40, 4, 96, 64, 5)


def test_soup_normals_and_specular(renderer, restated):
    _soup_case(renderer, restated, 6000, 20, 2, 80, 60, 9, edge=(0.05, 0.2), with_normals=True, specular=True)


def test_soup_with_spheres_extension(renderer, restated):
    """analytic spheres: no reference behaviour exists (parity unpinned); oracle = our restatement."""
    s, rs, cam, out, o = _soup_case(renderer, restated, 5000, 20, 2, 80, 60, 3, n_spheres=60, edge=(0.03, 0.1))
    assert (o.tri >= s.n_tris).any()


def test_coplanar_light_plane_and_eye_plane(renderer, restated):
    """Triangles exactly in the light's plane / through the eye: the filter's sign-ambiguous rows
    (slab rows and always-candidate rows) must not lose a single strict accept."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    s = scenes.coplanar_scene()
    W, H, seed = 120, 90, 13
    for eye in ((0, 1, 2.9), (0.4, 0.7, 2.5)):
        cam = Camera.for_frame(eye, (0, 1, 0), W, H)
        fid = hash_faceids(seed, W, H, s.faces_per_light)
        o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=fid)
        rs = renderer.upload(s)
        out = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True)
        _check_frame(out, W, H, o.tri, o.t, o.v, o.rgb, o.rgb8.reshape(-1, 3), occ=o.occ_tri)
        ex = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True, exhaustive_strict=True)
        assert ex.stats["filter_misses"] == 0 and ex.stats["pipeline_errors"] == 0
        assert np.array_equal(ex.rgb8, out.rgb8)


def test_soup_exhaustive_no_filter_misses(renderer):
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    s = scenes.soup_scene(3000, 12, 4, seed=8, edge=(0.02, 0.3))
    W, H = 64, 48
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, exhaustive_strict=True)
    assert b.stats["filter_misses"] == 0 and b.stats["pipeline_errors"] == 0
    assert np.array_equal(a.rgb8, b.rgb8) and np.array_equal(a.occ_tri, b.occ_tri) and np.array_equal(a.tri, b.tri)
    assert a.stats["strict_evals"] < b.stats["strict_evals"] / 20


def test_large_triangle_count_subset(renderer, restated):
    """200k triangles at 256x144 on the GPU; the oracle checks a random pixel subset."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    W, H, seed = 256, 144, 21
    s = scenes.soup_scene(200_000, 200, 4, seed=seed)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    out = renderer.trace(renderer.upload(s), cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True)
    fid = hash_faceids(seed, W, H, s.faces_per_light)
    idx = np.random.default_rng(0).choice(W * H, 192, replace=False)
    ph, pw = idx // W, idx % W
    o = restated.render_pixels(to_flat(s), cam.as_array(), W, H, pw, ph, fid[idx])
    k = (H - 1 - ph) * W + pw  # local (PPM-order) index
    assert np.array_equal(out.tri[k], o.tri)
    assert np.array_equal(bits(out.t[k]), bits(o.t))
    assert np.array_equal(out.occ_tri[k], o.occ_tri)
    assert np.array_equal(bits(out.rgb[k]), bits(o.rgb))
    assert np.array_equal(out.rgb8.reshape(-1, 3)[k], o.rgb8)


def test_bands_equal_whole_frame(renderer):
    """interleaved row bands rendered separately (what each rank does) == the whole frame, byte for byte"""
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    s = scenes.box_scene()
    W, H = 100, 77
    cam = Camera.for_frame((0, 1, 2.9), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    full = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4).rgb8
    for n, B in ((2, 8), (4, 8), (3, 5), (8, 16)):
        frame = np.zeros_like(full)
        for r in range(n):
            part = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, bands=(B, r, n)).rgb8
            rows = [pr for pr in range(H) if (pr // B) % n == r]
            assert part.shape[0] == len(rows)
            frame[rows] = part
        assert np.array_equal(frame, full)


def test_edge_cases(renderer):
    from esctp1raytracer_b200 import RNG_HASH, Camera, Scene, TracerError, scenes

    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), 16, 9)
    # empty scene: black frame (src/main.cpp:537-543 with no model)
    empty = Scene(np.array([0]), np.zeros((0, 3, 3), np.float32), np.zeros((0, 13), np.float32), np.zeros(0, np.int32))
    assert not renderer.trace(empty, cam, 16, 9).rgb8.any()
    # no light (models/cornell/water.obj): black frame
    s = scenes.box_scene()
    nolight = Scene(s.geom_tri_offset, s.tri_verts, s.geom_material, np.zeros(0, np.int32))
    out = renderer.trace(nolight, cam, 16, 9, debug=True)
    assert not out.rgb8.any() and (out.tri >= 0).any()
    # camera looking away: all rays miss
    away = Camera.for_frame((0, 1, 3), (0, 1, 6), 16, 9)
    out = renderer.trace(s, away, 16, 9, debug=True)
    assert (out.tri == -1).all() and not out.rgb8.any()
    # ragged sizes (not a multiple of anything), one-shot call
    assert renderer.trace(s, Camera.for_frame((0, 1, 2.9), (0, 1, 0), 37, 23), 37, 23).rgb8.shape == (23, 37, 3)
    with pytest.raises(TracerError):
        renderer.trace(s, cam, 1, 9)  # the reference divides by W-1


def test_idempotent_and_seed_sensitivity(renderer):
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    s = scenes.soup_scene(30000, 30, 4, seed=2)
    W, H = 128, 72
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=1).rgb8
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=1).rgb8
    c = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=2).rgb8
    assert np.array_equal(a, b) and not np.array_equal(a, c)


def test_fp32_peak_microbenchmark_runs(renderer):
    tf0, _ = renderer.fp32_peak(0, 3)
    tf1, _ = renderer.fp32_peak(1, 3)
    assert 10.0 < tf0 < 100.0 and 10.0 < tf1 < 100.0


def test_cli_host_flow_obj_to_ppm(renderer, restated, tmp_path):
    """The reference's whole flow (-m model.obj -v eye -l look -o out.ppm, src/main.cpp:417-695) through the C++ CLI:
    our OBJ loader -> camera -> GPU render (std::mt19937 seeded) -> P3 writer, checked against the oracle."""
    import subprocess

    from conftest import ROOT
    from esctp1raytracer_b200 import Scene, scenes

    s = scenes.box_scene()
    from conftest import write_obj

    obj = tmp_path / "box.obj"
    write_obj(s, obj)
    loaded = Scene.load_obj(str(obj))
    assert np.array_equal(bits(loaded.tri_verts), bits(s.tri_verts)) and np.array_equal(loaded.light_geom, s.light_geom)
    assert np.array_equal(bits(loaded.geom_material), bits(s.geom_material))
    out = tmp_path / "out.ppm"
    W, H, seed = 96, 72, 31
    cli = os.path.join(ROOT, "esctp1raytracer_b200", "tracer_cli.bin")
    r = subprocess.run([cli, "-m", str(obj), "-v", "0,1,2.9", "-l", "0,1,0", "-w", f"{W},{H}", "--seed", str(seed), "-o", str(out)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Duration" in r.stderr and "Rendered image in" in r.stdout
    tok = out.read_text().split()
    assert tok[:4] == ["P3", str(W), str(H), "255"]
    got = np.array(tok[4:], dtype=np.int64).reshape(H, W, 3)
    o = restated.render(to_flat(loaded), restated.camera((0, 1, 2.9), (0, 1, 0), W, H), W, H, seed=seed)
    assert np.array_equal(got, o.rgb8)
    out2 = tmp_path / "out_cull.ppm"  # the optional bundle-cull mode writes the same file
    r = subprocess.run([cli, "-m", str(obj), "-v", "0,1,2.9", "-l", "0,1,0", "-w", f"{W},{H}", "--seed", str(seed), "--cull", "-o",
                        str(out2)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert out2.read_bytes() == out.read_bytes()


def test_multisample_jitter_extension(renderer, restated):
    """n x n stratified jittered samples per pixel (BASELINE config 5; no reference code: parity unpinned,
    oracle = our restatement).  Same strict arithmetic on both sides -> bit-equal mean colour."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, TracerError, scenes

    s = scenes.soup_scene(3000, 12, 2, seed=4, edge=(0.05, 0.2), n_spheres=10)
    W, H, seed = 64, 40, 17
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    for spp in (4, 9):
        n = int(round(spp ** 0.5))
        rgb, rgb8 = restated.render_spp(to_flat(s), cam.as_array(), W, H, seed, n)
        out = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, samples_per_pixel=spp, debug=True)
        assert np.array_equal(bits(out.rgb), bits(_to_ppm_order(rgb, W, H)))
        assert np.array_equal(out.rgb8, rgb8)
        assert out.stats["n_primary_rays"] == W * H * spp
        # jittered rays of a thread share a MEAN q in the span sweep (mean q + |B| * spread): still a necessary condition
        ex = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, samples_per_pixel=spp, debug=True, exhaustive_strict=True)
        assert ex.stats["filter_misses"] == 0 and ex.stats["pipeline_errors"] == 0
        assert np.array_equal(bits(out.rgb), bits(ex.rgb)) and np.array_equal(out.rgb8, ex.rgb8)
        for R in (2, 4, 8, 16):
            o2 = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, samples_per_pixel=spp, debug=True, rays_per_thread=R)
            assert np.array_equal(bits(out.rgb), bits(o2.rgb)), R
    # frames too small for the span rows' parameter range keep the three-row sweep (every ray its own q)
    Ws, Hs = 12, 9
    cams = Camera.for_frame((0, 1, 3), (0, 1, 0), Ws, Hs)
    rgb, rgb8 = restated.render_spp(to_flat(s), cams.as_array(), Ws, Hs, seed, 2)
    out = renderer.trace(rs, cams, Ws, Hs, rng_mode=RNG_HASH, seed=seed, samples_per_pixel=4, debug=True)
    assert np.array_equal(bits(out.rgb), bits(_to_ppm_order(rgb, Ws, Hs))) and np.array_equal(out.rgb8, rgb8)
    ex = renderer.trace(rs, cams, Ws, Hs, rng_mode=RNG_HASH, seed=seed, samples_per_pixel=4, debug=True, exhaustive_strict=True)
    assert ex.stats["filter_misses"] == 0 and np.array_equal(out.rgb8, ex.rgb8)
    with pytest.raises(TracerError):
        renderer.trace(rs, cam, W, H, samples_per_pixel=5)  # not a square


def _same_frames(a, b):
    assert np.array_equal(a.rgb8, b.rgb8)
    assert np.array_equal(a.tri, b.tri) and np.array_equal(bits(a.t), bits(b.t)) and np.array_equal(bits(a.v), bits(b.v))
    assert np.array_equal(a.occ_tri, b.occ_tri) and np.array_equal(bits(a.rgb), bits(b.rgb))


@pytest.mark.parametrize("name", golden_names())
def test_bundle_cull_golden(renderer, name):
    """OPTIONAL bundle-cull mode against the reference's own frames."""
    from esctp1raytracer_b200 import RNG_EXPLICIT

    fs, fr = load_golden(name)
    W, H = fr["W"], fr["H"]
    out = renderer.trace(renderer.upload(to_scene(fs)), _cam(fr), W, H, rng_mode=RNG_EXPLICIT, faceid=fr["faceid"], debug=True,
                         bundle_cull=True)
    _check_frame(out, W, H, fr["tri"], fr["t"], fr["v"], fr["rgb"], fr["q"])


def test_bundle_cull_identical_to_default(renderer):
    """hierarchical evaluation of the same filter: every debug output bit-identical to the default mode"""
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    cases = [
        (scenes.soup_scene(20000, 40, 4, seed=5), 96, 64, (0, 1, 3)),
        (scenes.soup_scene(6000, 20, 2, seed=9, edge=(0.05, 0.2), with_normals=True, specular=True, n_spheres=30), 80, 60, (0, 1, 3)),
        (scenes.coplanar_scene(), 120, 90, (0, 1, 2.9)),
        (scenes.soup_scene(60000, 60, 4, seed=1), 333, 187, (0.3, 1.2, 2.7)),  # ragged tile edges
    ]
    for s, W, H, eye in cases:
        cam = Camera.for_frame(eye, (0, 1, 0), W, H)
        rs = renderer.upload(s)
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True)
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bundle_cull=True)
        _same_frames(a, b)
        assert b.stats["tests_shadow_ref"] == a.stats["tests_shadow_ref"] and b.stats["n_shadow_rays"] == a.stats["n_shadow_rays"]
        c = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bundle_cull=2)  # streaming form (fall-back)
        _same_frames(a, c)
        d = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bundle_cull=3)  # auto (picks the default sweeps here)
        _same_frames(a, d)
    # bands and multi-sample in cull mode
    s, W, H = cases[0][0], 100, 77
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    full = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4).rgb8
    frame = np.zeros_like(full)
    for r in range(3):
        part = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, bands=(8, r, 3), bundle_cull=True).rgb8
        frame[[pr for pr in range(H) if (pr // 8) % 3 == r]] = part
    assert np.array_equal(frame, full)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, samples_per_pixel=4)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=4, samples_per_pixel=4, bundle_cull=True)
    assert np.array_equal(a.rgb8, b.rgb8)


def test_full_size_c4_frame(renderer, restated):
    """BASELINE.json configs[3] at full size (1M triangles + 1k spheres, 3840x2160, 4 lights).  The oracle
    needs ~0.1 core-seconds per pixel here, so it checks a random pixel subset bit for bit; the whole frame is
    checked through a size-independent property: the default sweep and the bundle-cull mode — two different
    evaluations of the filter with different work decompositions, ray orders and merge paths — must produce
    byte-identical frames, hit ids, occluders and float accumulators."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True, bundle_cull=True)
    _same_frames(a, b)
    assert a.stats["n_primary_rays"] == W * H and a.stats["tests_primary"] == W * H * 1_000_000
    assert (a.tri >= 0).sum() * 4 == a.stats["n_shadow_rays"]
    fid = hash_faceids(seed, W, H, s.faces_per_light)
    idx = np.random.default_rng(1).choice(W * H, 96, replace=False)
    ph, pw = idx // W, idx % W
    o = restated.render_pixels(to_flat(s), cam.as_array(), W, H, pw, ph, fid[idx], n_threads=os.cpu_count() or 1)
    k = (H - 1 - ph) * W + pw
    assert np.array_equal(a.tri[k], o.tri)
    assert np.array_equal(bits(a.t[k]), bits(o.t))
    assert np.array_equal(a.occ_tri[k], o.occ_tri)
    assert np.array_equal(bits(a.rgb[k]), bits(o.rgb))
    assert np.array_equal(a.rgb8.reshape(-1, 3)[k], o.rgb8)


def test_render_frame_is_ordered_on_torchs_stream(renderer):
    """dist.render_frame hands the library torch's current stream; the legacy default stream must go in as
    cudaStreamLegacy (0x1), never as 0 (= the library's own stream, unordered with torch's allocations and NCCL)."""
    import torch

    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes
    from esctp1raytracer_b200 import dist as tdist

    assert tdist.torch_stream_handle() != 0
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        assert tdist.torch_stream_handle() == side.cuda_stream
    s = scenes.soup_scene(3000, 10, 2, seed=2)
    W, H = 96, 64
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    want = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=5).rgb8
    for _ in range(3):  # back to back, no synchronize in between
        a, _ = tdist.render_frame(renderer, rs, cam, W, H, seed=5)
        b, _ = tdist.render_frame(renderer, rs, cam, W, H, seed=5, bundle_cull=True)
    assert np.array_equal(a.cpu().numpy(), want) and np.array_equal(b.cpu().numpy(), want)


def test_bundle_cull_falls_back_to_streaming_when_keys_do_not_fit(renderer):
    """two-phase mode: when phase A's survivor keys would not fit their buffer the sweep must fall back to the
    streaming form and still produce the default mode's frame (the buffer limit is faked with TRACER_L0_CAP)."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    s = scenes.soup_scene(20000, 40, 3, seed=6)
    W, H = 96, 64
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True)
    os.environ["TRACER_L0_CAP"] = "100"
    try:
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bundle_cull=1)
    finally:
        del os.environ["TRACER_L0_CAP"]
    _same_frames(a, b)


def test_shadow_sweeps_with_shared_q_terms_never_miss(renderer, restated):
    """Default-mode shadow sweeps order each (light vertex, face) list by q and evaluate the 8 consecutive rays of a
    thread with one q-term per edge row (qbar + |B|*qdelta).  That must stay a necessary condition: exhaustive mode
    strict-tests every pair and counts accepts the filter would have lost (0), frames equal the oracle, and the
    order-preserving compaction is exercised with many chunks."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    for s, W, H, chunks in ((scenes.soup_scene(30000, 30, 4, seed=12, edge=(0.02, 0.25)), 160, 100, 24),
                            (scenes.coplanar_scene(), 120, 90, 5),
                            (scenes.soup_scene(9000, 9, 3, seed=4, with_normals=True, specular=True, n_spheres=11), 75, 49, 0)):
        cam = Camera.for_frame((0, 1, 2.9), (0, 1, 0), W, H)
        rs = renderer.upload(s)
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=7, debug=True, shadow_chunks=chunks)
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=7, debug=True, shadow_chunks=chunks, exhaustive_strict=True)
        assert b.stats["filter_misses"] == 0 and b.stats["pipeline_errors"] == 0
        _same_frames(a, b)
        o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(7, W, H, s.faces_per_light))
        _check_frame(a, W, H, o.tri, o.t, o.v, o.rgb, o.rgb8.reshape(-1, 3), occ=o.occ_tri)
        assert a.stats["tests_shadow_ref"] == o.n_tests[1]


def test_big_light_tables_are_batched_within_a_budget(renderer, restated):
    """ADVICE r1 (medium): the 6 cube-face filter tables per light vertex used to be allocated for ALL light vertices up
    front, so an emissive mesh could be refused outright.  They now live in a budgeted number of slots that each light's
    vertices go through batch by batch (TRACER_TABLE_SLOTS fakes a tiny budget): same frame as with resident tables."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    s = scenes.soup_scene(12000, 12, 3, seed=21, n_spheres=4)
    W, H = 112, 70
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    a = renderer.trace(renderer.upload(s), cam, W, H, rng_mode=RNG_HASH, seed=6, debug=True)
    os.environ["TRACER_TABLE_SLOTS"] = "1"
    try:
        rs = renderer.upload(s)  # the budget is taken at scene creation
    finally:
        del os.environ["TRACER_TABLE_SLOTS"]
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=6, debug=True)
    _same_frames(a, b)
    c = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=6, debug=True, bundle_cull=True)  # falls back to the default sweeps
    _same_frames(a, c)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(6, W, H, s.faces_per_light))
    _check_frame(b, W, H, o.tri, o.t, o.v, o.rgb, o.rgb8.reshape(-1, 3), occ=o.occ_tri)


def test_bundle_cull_overflow_rerenders_in_default_mode(renderer):
    """ADVICE r1 (low): a candidate-buffer overflow in the optional mode used to reject the frame after all the work;
    now the frame is rendered again by the default sweeps (TRACER_CAND_CAP fakes a tiny buffer)."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    s = scenes.soup_scene(20000, 40, 3, seed=6)
    W, H = 96, 64
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True)
    os.environ["TRACER_CAND_CAP"] = "1000"
    try:
        for mode in (1, 2):
            b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, bundle_cull=mode)
            _same_frames(a, b)
            assert b.stats["flop_primary"] > 0  # the statistics are the default sweeps'
    finally:
        del os.environ["TRACER_CAND_CAP"]


def test_span_sweeps_every_rays_per_thread_variant(renderer, restated):
    """The default sweeps evaluate the filter in SPAN form (two lower + two upper bounds of p per triangle, sweep.cuh).
    Every rays-per-thread instantiation of the closest-hit sweep (2..32; screen tiles of different shapes) must give the
    oracle's frame, and exhaustive mode — which also checks the hot loop's own group verdicts — must find no accept the
    filter would have lost."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    s = scenes.soup_scene(12000, 12, 3, seed=21, edge=(0.02, 0.4))
    W, H = 300, 70  # wider than one 256-pixel tile row of the 32-ray variant, ragged at both edges
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(9, W, H, s.faces_per_light))
    for R in (0, 2, 4, 8, 16, 24, 32):
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=9, debug=True, rays_per_thread=R)
        _check_frame(a, W, H, o.tri, o.t, o.v, o.rgb, o.rgb8.reshape(-1, 3), occ=o.occ_tri)
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=9, debug=True, rays_per_thread=R, exhaustive_strict=True)
        assert b.stats["filter_misses"] == 0 and b.stats["pipeline_errors"] == 0, R
        _same_frames(a, b)


def test_span_rows_with_huge_and_degenerate_triangles(renderer, restated):
    """Span rows divide each edge row by its p-coefficient.  Stress what that could break: triangles that span tens of
    degrees as seen from the eye and from the lights (cones that reach around the parametrisation plane: three bounds on
    one side, one is dropped), edges parallel to the p axis (coefficient ~ 0), zero-area and needle triangles, triangles
    through the eye's plane.  Frames equal the oracle; exhaustive mode finds no filter miss."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    rng = np.random.default_rng(5)
    s = scenes.soup_scene(200, 6, 2, seed=31, edge=(0.2, 1.5))  # big triangles all around the eye and the lights
    v = s.tri_verts.reshape(-1, 3, 3).copy()  # triangles 0-3: floor and wall, 4-7: the two lights (left alone)
    for i in range(8, 40):  # axis-aligned edges: rows whose p- or q-coefficient vanishes
        v[i, 1] = v[i, 0] + np.array([rng.uniform(0.2, 2.0), 0.0, 0.0], np.float32)
        v[i, 2] = v[i, 0] + np.array([0.0, rng.uniform(0.2, 2.0), 0.0], np.float32)
    for i in range(40, 60):  # needles and zero-area triangles
        v[i, 1] = v[i, 0] + np.float32(1e-6) * rng.normal(size=3).astype(np.float32)
        v[i, 2] = v[i, 0] + (v[i, 1] - v[i, 0]) * np.float32(2.0) if i % 2 else v[i, 0]
    for i in range(60, 90):  # through the plane of the eye (z = 3): the cone wraps around the image plane
        v[i, 0, 2], v[i, 1, 2], v[i, 2, 2] = 2.0, 4.5, 3.0
    s.tri_verts = np.ascontiguousarray(v, np.float32)
    for (W, H, eye, look) in ((160, 90, (0, 1, 3), (0, 1, 0)), (97, 61, (0.3, 0.8, 0.5), (0.1, 1.0, -1.0))):
        cam = Camera.for_frame(eye, look, W, H)
        rs = renderer.upload(s)
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=2, debug=True)
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=2, debug=True, exhaustive_strict=True)
        assert b.stats["filter_misses"] == 0 and b.stats["pipeline_errors"] == 0
        _same_frames(a, b)
        o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(2, W, H, s.faces_per_light))
        _check_frame(a, W, H, o.tri, o.t, o.v, o.rgb, o.rgb8.reshape(-1, 3), occ=o.occ_tri)
        # the filter must still filter
        assert a.stats["strict_evals"] < 0.5 * b.stats["strict_evals"]
