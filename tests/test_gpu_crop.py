"""Crop windows (Renderer.trace(..., crop=(x, y, w, h)), opts.crop_*): a window of a frame is bit for bit the same pixels of
the whole frame, in every mode and RNG mode: packed bytes, hit ids, t, v, first occluders and the float accumulator."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT, bits, golden_names, load_golden, to_scene, write_obj

pytestmark = pytest.mark.gpu

W, H = 300, 90  # a multiple of no tile width
EYE, LOOK = (0.0, 1.0, 3.0), (0.0, 1.0, 0.0)
# (x, y, w, h) in PPM coordinates: centre, 1 x 1, the bottom-right corner (a seeded crop's covering rows are the whole
# frame), one row, one column
CROPS = [(117, 31, 61, 23), (0, 0, 1, 1), (W - 5, H - 3, 5, 3), (0, 40, W, 1), (150, 0, 1, H)]
# every edge, widths that are no multiple of 64, 128 or 256 and one under a tile, and the whole frame
SHAPES = [(0, 0, 63, 9), (W - 127, 0, 127, 12), (0, H - 7, 129, 7), (W - 255, H - 11, 255, 11), (13, 20, 257, 50),
          (W - 1, 0, 1, H), (0, H - 1, W, 1), (101, 44, 5, 2), (0, 0, W, H)]


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


@pytest.fixture(scope="module")
def soup():
    from esctp1raytracer_b200 import scenes

    return scenes.soup_scene(20000, 40, 4, seed=5, n_spheres=20)


def _cam(w=W, h=H):
    from esctp1raytracer_b200 import Camera

    return Camera.for_frame(EYE, LOOK, w, h)


def _faceids(scene, seed=3):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(0, f, W * H) for f in scene.faces_per_light], 1).astype(np.int32)


def _same_pixels(crop, full, window, w=W, h=H):
    """crop frame equals the window of the full frame: bytes, hit ids, t / v bits, first occluders, float accumulator"""
    x, y, cw, ch = window
    assert crop.rgb8.shape == (ch, cw, 3)
    assert np.array_equal(crop.rgb8, full.rgb8[y:y + ch, x:x + cw]), ("packed bytes differ", window)

    def cut(a):
        return a.reshape((h, w) + a.shape[1:])[y:y + ch, x:x + cw].reshape((ch * cw,) + a.shape[1:])

    assert np.array_equal(crop.tri, cut(full.tri)), ("hit ids differ", window)
    assert np.array_equal(bits(crop.t), bits(cut(full.t))) and np.array_equal(bits(crop.v), bits(cut(full.v))), window
    assert np.array_equal(crop.occ_tri, cut(full.occ_tri)), ("first occluders differ", window)
    assert np.array_equal(bits(crop.rgb), bits(cut(full.rgb))), ("float accumulator differs", window)


RNG = [
    dict(rng_mode=0, seed=11),
    dict(rng_mode=1, seed=12),
    dict(rng_mode=2),
    dict(rng_mode=0, seed=13, samples_per_pixel=4),
    dict(rng_mode=2, samples_per_pixel=4),
]
MODES = [dict(), dict(bundle_cull=1), dict(bundle_cull=2), dict(bundle_cull=3), dict(bvh=True)]


@pytest.mark.parametrize("mode", range(len(MODES)))
@pytest.mark.parametrize("rng", range(len(RNG)))
def test_crop_equals_full_frame(renderer, soup, mode, rng):
    kw = dict(RNG[rng], **MODES[mode])
    if kw["rng_mode"] == 2:
        kw["faceid"] = _faceids(soup)
    rs = renderer.upload(soup)
    full = renderer.trace(rs, _cam(), W, H, debug=True, **kw)
    for window in CROPS:
        crop = renderer.trace(rs, _cam(), W, H, debug=True, crop=window, **kw)
        _same_pixels(crop, full, window)
        assert crop.stats["n_pixels"] == window[2] * window[3]


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("rays_per_thread", [0, 64])
def test_crop_shapes(renderer, soup, rng_mode, rays_per_thread):
    kw = dict(rng_mode=rng_mode, seed=7, rays_per_thread=rays_per_thread)
    rs = renderer.upload(soup)
    full = renderer.trace(rs, _cam(), W, H, debug=True, **kw)
    for window in SHAPES:
        _same_pixels(renderer.trace(rs, _cam(), W, H, debug=True, crop=window, **kw), full, window)


@pytest.mark.parametrize("mode", [dict(), dict(bundle_cull=1)])
@pytest.mark.parametrize("rng_mode", [0, 1])
def test_exhaustive_strict_crop(renderer, soup, mode, rng_mode):
    rs = renderer.upload(soup)
    kw = dict(rng_mode=rng_mode, seed=21, exhaustive_strict=True, **mode)
    full = renderer.trace(rs, _cam(), W, H, debug=True, **kw)
    for window in CROPS[:3]:
        crop = renderer.trace(rs, _cam(), W, H, debug=True, crop=window, **kw)
        _same_pixels(crop, full, window)
        assert crop.stats["filter_misses"] == 0 and crop.stats["pipeline_errors"] == 0


def test_whole_frame_crop_is_the_frame(renderer, soup):
    """a window of the whole frame: the uncropped call's bytes; with hashed faceIDs its work too, seeded one gather more"""
    rs = renderer.upload(soup)
    counters = ("n_pixels", "n_primary_rays", "n_shadow_rays", "tests_primary", "tests_shadow", "tests_shadow_ref")
    for rng_mode, extra in ((0, 0), (1, 1)):
        renderer.trace(rs, _cam(), W, H, rng_mode=rng_mode, seed=5)  # the lazily built shadow tables, before the compared frames
        full = renderer.trace(rs, _cam(), W, H, rng_mode=rng_mode, seed=5, debug=True)
        crop = renderer.trace(rs, _cam(), W, H, rng_mode=rng_mode, seed=5, debug=True, crop=(0, 0, W, H))
        _same_pixels(crop, full, (0, 0, W, H))
        for key in counters:
            assert crop.stats[key] == full.stats[key], (rng_mode, key)
        assert crop.stats["kernel_launches"] == full.stats["kernel_launches"] + extra, rng_mode


def test_seeded_crop_counts_its_covering_rows(renderer, soup):
    rs = renderer.upload(soup)
    window = (40, 20, 30, 10)
    crop = renderer.trace(rs, _cam(), W, H, rng_mode=1, seed=5, crop=window)
    assert crop.stats["n_pixels"] == 300 and crop.stats["n_primary_rays"] == W * 30
    hashed = renderer.trace(rs, _cam(), W, H, rng_mode=0, seed=5, crop=window)
    assert hashed.stats["n_primary_rays"] == 300 and hashed.stats["tests_primary"] < crop.stats["tests_primary"]


@pytest.mark.parametrize("name", golden_names())
def test_golden_crops(renderer, name):
    """windows of the reference's own frames, with its seed and with its faceIDs"""
    from esctp1raytracer_b200 import RNG_EXPLICIT, RNG_MT19937, Camera

    fs, fr = load_golden(name)
    w, h = fr["W"], fr["H"]
    cam = Camera.for_frame(fr["eye"], fr["look"], w, h)
    rs = renderer.upload(to_scene(fs))

    def ppm(a):  # image index order (h*W+w) -> PPM row order
        return a.reshape(h, w, *a.shape[1:])[::-1].reshape(a.shape)

    want = dict(rgb8=np.asarray(fr["q"], np.uint8).reshape(h, w, 3), tri=ppm(fr["tri"]), t=ppm(fr["t"]), v=ppm(fr["v"]),
                rgb=ppm(np.asarray(fr["rgb"], np.float32).reshape(h * w, 3)))
    windows = [(w // 3, h // 3, w // 3 + 1, h // 4), (w - 17, h - 9, 17, 9), (0, h // 2, w, 1), (5, 0, 1, h)]
    for kw in (dict(rng_mode=RNG_MT19937, seed=fr["seed"]), dict(rng_mode=RNG_EXPLICIT, faceid=fr["faceid"])):
        for x, y, cw, ch in windows:
            out = renderer.trace(rs, cam, w, h, debug=True, crop=(x, y, cw, ch), **kw)

            def cut(a):
                return a.reshape((h, w) + a.shape[1:])[y:y + ch, x:x + cw].reshape((ch * cw,) + a.shape[1:])

            assert np.array_equal(out.rgb8, want["rgb8"][y:y + ch, x:x + cw]), ("PPM bytes differ", kw["rng_mode"], (x, y))
            assert np.array_equal(out.tri, cut(want["tri"])), "hit ids differ"
            assert np.array_equal(bits(out.t), bits(cut(want["t"]))) and np.array_equal(bits(out.v), bits(cut(want["v"])))
            assert np.array_equal(bits(out.rgb), bits(cut(want["rgb"]))), "float accumulator differs"


def test_seeded_crop_after_candidate_overflow(renderer, soup, monkeypatch):
    """a bundle-cull covering pass whose candidates overflow renders again before its row counts are used"""
    rs = renderer.upload(soup)
    full = renderer.trace(rs, _cam(), W, H, rng_mode=1, seed=3, debug=True)
    monkeypatch.setenv("TRACER_CAND_CAP", "1000")
    for mode in (1, 2):
        for window in ((117, 31, 61, 23), (W - 5, H - 3, 5, 3)):
            crop = renderer.trace(rs, _cam(), W, H, rng_mode=1, seed=3, debug=True, bundle_cull=mode, crop=window)
            assert crop.stats["flop_primary"] > 0  # rendered again by the default sweeps
            _same_pixels(crop, full, window)


def test_crop_after_scene_update(renderer, soup):
    from esctp1raytracer_b200 import Scene

    rs = renderer.upload(soup)
    renderer.trace(rs, _cam(), W, H, rng_mode=1, seed=6)  # tables built before the move
    g = 7
    a, b = int(soup.geom_tri_offset[g]), int(soup.geom_tri_offset[g + 1])
    moved = soup.tri_verts.copy()
    moved[a:b] += np.float32([0.3, -0.2, 0.1])
    rs.update(tri_verts=moved[a:b], first_tri=a)
    fresh = renderer.upload(Scene(soup.geom_tri_offset, moved, soup.geom_material, soup.light_geom, sphere_cr=soup.sphere_cr,
                                  sphere_material=soup.sphere_material))
    for kw in (dict(rng_mode=1, seed=6), dict(rng_mode=0, seed=6, bvh=True)):
        full = renderer.trace(fresh, _cam(), W, H, debug=True, **kw)
        for window in CROPS[:3]:
            _same_pixels(renderer.trace(rs, _cam(), W, H, debug=True, crop=window, **kw), full, window)


def test_one_shot_crop(renderer, soup):
    rs = renderer.upload(soup)
    for kw in (dict(rng_mode=0, seed=9), dict(rng_mode=1, seed=9)):
        full = renderer.trace(rs, _cam(), W, H, debug=True, **kw)
        window = (117, 31, 61, 23)
        _same_pixels(renderer.trace(soup, _cam(), W, H, debug=True, crop=window, **kw), full, window)


def test_device_output_and_caller_out(renderer, soup):
    torch = pytest.importorskip("torch")
    rs = renderer.upload(soup)
    window = (117, 31, 61, 23)
    want = renderer.trace(rs, _cam(), W, H, seed=8, crop=window)
    buf = torch.zeros(61 * 23 * 3, dtype=torch.uint8, device="cuda")
    renderer.trace(rs, _cam(), W, H, seed=8, crop=window, out_device_ptr=buf.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(buf.cpu().numpy().reshape(want.rgb8.shape), want.rgb8)
    out = np.zeros((23, 61, 3), np.uint8)
    assert renderer.trace(rs, _cam(), W, H, seed=8, crop=window, out=out).rgb8 is out
    assert np.array_equal(out, want.rgb8)


def test_refusals(renderer, soup):
    from esctp1raytracer_b200 import MultiRenderer, Renderer, _lib

    rs = renderer.upload(soup)
    cam = _cam()
    out = np.zeros(W * H * 3, np.uint8)
    dst = out.ctypes.data_as(C.c_void_p)

    def opts(**kw):
        o = _lib.RenderOpts()
        o.struct_size = C.sizeof(_lib.RenderOpts)
        for k, v in kw.items():
            setattr(o, k, v)
        return C.byref(o)

    def scene_call(**kw):
        return renderer.lib.tracer_cuda_render_scene(rs.handle, C.byref(cam.c), W, H, opts(**kw), dst)

    bad = [dict(crop_x=1), dict(crop_w=5), dict(crop_w=5, crop_h=-1), dict(crop_x=-1, crop_w=5, crop_h=5),
           dict(crop_x=W - 4, crop_w=5, crop_h=5), dict(crop_y=H - 4, crop_w=5, crop_h=5), dict(crop_w=W + 1, crop_h=1),
           dict(crop_x=2 ** 31 - 1, crop_w=5, crop_h=5), dict(crop_w=5, crop_h=5, band_rows=8, band_index=0, band_count=2)]
    for kw in bad:
        assert scene_call(**kw) == -1, kw
    cs = soup.c_struct()
    assert renderer.lib.tracer_cuda_render(C.byref(cs), C.byref(cam.c), W, H, opts(crop_x=-1, crop_w=5, crop_h=5), dst) == -1
    carr = (_lib.CameraC * 2)(cam.c, cam.c)
    assert renderer.lib.tracer_cuda_render_views(rs.handle, carr, 2, W, H, opts(crop_w=5, crop_h=5), dst) == -1
    assert renderer.lib.tracer_cuda_render_views(rs.handle, carr, 1, W, H, opts(crop_w=5, crop_h=5), dst) == -1
    # an older caller (struct_size up to row_hits_user) renders the whole frame whatever lies past its struct
    o = _lib.RenderOpts()
    o.struct_size, o.rng_mode, o.seed = _lib.RenderOpts.crop_x.offset, 0, 4
    o.crop_x, o.crop_w, o.crop_h = 3, 5, 5
    assert renderer.lib.tracer_cuda_render_scene(rs.handle, C.byref(cam.c), W, H, C.byref(o), dst) == 0
    assert np.array_equal(out.reshape(H, W, 3), renderer.trace(rs, cam, W, H, seed=4).rgb8)
    for kw in (dict(crop=(0, 0, 0, 0)), dict(crop=(W - 4, 0, 5, 5)), dict(crop=(0, 0, 5, 5), bands=(8, 0, 2)),
               dict(crop=(0, 0, 5, 5), out=np.zeros((5, 6, 3), np.uint8))):
        with pytest.raises(ValueError):
            renderer.trace(rs, cam, W, H, **kw)
    with pytest.raises(TypeError):
        renderer.trace_views(rs, [cam], W, H, crop=(0, 0, 5, 5))
    # the multi-GPU calls, also with one GPU (where tracer_cuda_render_scene_multi forwards to the single-GPU call)
    m = MultiRenderer(1)
    ms = m.upload(soup)
    assert m.lib.tracer_cuda_render_scene_multi(ms.handle, C.byref(cam.c), W, H, opts(crop_w=5, crop_h=5), dst) == -1
    assert m.lib.tracer_cuda_render_multi(C.byref(cs), C.byref(cam.c), W, H, opts(crop_w=5, crop_h=5), dst) == -1
    assert b"crop" in m.lib.tracer_cuda_last_error()
    with pytest.raises(TypeError):
        m.trace(ms, cam, W, H, crop=(0, 0, 5, 5))
    ms.close()
    Renderer(0)  # device 0 is the current context again, as for the module's renderer
    after = renderer.trace(rs, cam, W, H, seed=3, debug=True, crop=(10, 10, 20, 20))
    _same_pixels(after, renderer.trace(rs, cam, W, H, seed=3, debug=True), (10, 10, 20, 20))


def _read_ppm(path):
    data = open(path, "rb").read()
    parts = data.split(b"\n", 3)
    assert parts[0] == b"P6"
    w, h = (int(x) for x in parts[1].split())
    return np.frombuffer(parts[3], np.uint8).reshape(h, w, 3)


def test_cli_crop(soup, tmp_path):
    obj = tmp_path / "soup.obj"
    write_obj(soup, obj)
    cli = os.path.join(ROOT, "esctp1raytracer_b200", "tracer_cli.bin")
    base = [cli, "-m", str(obj), "-v", "0,1,3", "-l", "0,1,0", "-w", f"{W},{H}", "--seed", "7", "--p6"]
    x, y, cw, ch = 117, 31, 61, 23
    for extra in ([], ["--rng", "hash"], ["--cull"], ["--bvh"]):
        full, part = tmp_path / "full.ppm", tmp_path / "crop.ppm"
        r = subprocess.run(base + extra + ["-o", str(full)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        r = subprocess.run(base + extra + ["--crop", f"{x},{y},{cw},{ch}", "-o", str(part)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        got = _read_ppm(part)
        assert got.shape == (ch, cw, 3)
        assert np.array_equal(got, _read_ppm(full)[y:y + ch, x:x + cw]), extra
    r = subprocess.run(base + ["--crop", f"{W - 4},0,5,5"], capture_output=True, text=True)
    assert r.returncode != 0 and "crop window" in r.stderr
