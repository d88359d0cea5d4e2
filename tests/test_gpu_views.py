"""Several cameras of one resident scene in one call (Renderer.trace_views, tracer_cuda_render_views): every view is bit for
bit the frame a single render of that camera gives."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT, bits, golden_names, load_golden, to_scene, write_obj

pytestmark = pytest.mark.gpu

W, H = 130, 70  # a multiple of no tile width
LOOK = (0.0, 1.0, 0.0)
# one eye inside the scene box, one far outside it: the call's common reach bound differs from every view's own
EYES = [(0.0, 1.0, 3.0), (2.5, 1.6, 2.0), (0.2, 1.0, 0.3), (-40.0, 9.0, 60.0), (-1.5, 0.4, -2.8)]
STAT_SUMS = ("n_pixels", "n_primary_rays", "n_shadow_rays", "tests_shadow_ref")


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


@pytest.fixture(scope="module")
def soup():
    from esctp1raytracer_b200 import scenes

    return scenes.soup_scene(20000, 40, 4, seed=5, n_spheres=20)


def _cams(eyes, w=W, h=H):
    from esctp1raytracer_b200 import Camera

    return [Camera.for_frame(e, LOOK, w, h) for e in eyes]


def _faceids(scene, n_views, seed=3):
    rng = np.random.default_rng(seed)
    F = scene.faces_per_light
    return np.stack([np.stack([rng.integers(0, f, W * H) for f in F], 1) for _ in range(n_views)]).astype(np.int32)


def _same_frame(a, b, v=None):
    """view v of batch frame a equals single frame b: packed bytes, hit ids, t/v bits, first occluders, float accumulator"""
    pick = (lambda x: x[v]) if v is not None else (lambda x: x)
    assert np.array_equal(pick(a.rgb8), b.rgb8), "packed bytes differ"
    assert np.array_equal(pick(a.tri), b.tri), "hit ids differ"
    assert np.array_equal(bits(pick(a.t)), bits(b.t)) and np.array_equal(bits(pick(a.v)), bits(b.v)), "t / v differ"
    assert np.array_equal(pick(a.occ_tri), b.occ_tri), "first occluders differ"
    assert np.array_equal(bits(pick(a.rgb)), bits(b.rgb)), "float accumulator differs"


def _batch_vs_singles(renderer, rs, eyes, **kw):
    from esctp1raytracer_b200 import RNG_EXPLICIT

    cams = _cams(eyes)
    fid = kw.pop("faceid", None)
    batch = renderer.trace_views(rs, cams, W, H, debug=True, faceid=fid, **kw)
    assert batch.rgb8.shape == (len(cams), H, W, 3) and batch.tri.shape == (len(cams), H * W)
    singles = []
    for v, cam in enumerate(cams):
        one = renderer.trace(rs, cam, W, H, debug=True, faceid=None if fid is None else fid[v], **kw)
        _same_frame(batch, one, v)
        singles.append(one)
    for key in STAT_SUMS:
        assert batch.stats[key] == sum(s.stats[key] for s in singles), key
    if not kw.get("bvh"):
        assert batch.stats["tests_primary"] == sum(s.stats["tests_primary"] for s in singles)
    if kw.get("rng_mode") == RNG_EXPLICIT:
        assert fid is not None
    return batch


MODES = [
    dict(rng_mode=0, seed=11),
    dict(rng_mode=1, seed=12),
    dict(rng_mode=2),
    dict(rng_mode=0, seed=13, samples_per_pixel=4),
    dict(rng_mode=2, samples_per_pixel=4),
]


@pytest.mark.parametrize("bvh", [False, True])
@pytest.mark.parametrize("mode", range(len(MODES)))
def test_batch_equals_single_renders(renderer, soup, mode, bvh):
    kw = dict(MODES[mode])
    if kw["rng_mode"] == 2:
        kw["faceid"] = _faceids(soup, len(EYES))
    rs = renderer.upload(soup)
    _batch_vs_singles(renderer, rs, EYES, bvh=bvh, **kw)


@pytest.mark.parametrize("rng_mode", [0, 1])
def test_exhaustive_strict_batch(renderer, soup, rng_mode):
    rs = renderer.upload(soup)
    b = _batch_vs_singles(renderer, rs, EYES, rng_mode=rng_mode, seed=21, exhaustive_strict=True)
    assert b.stats["filter_misses"] == 0 and b.stats["pipeline_errors"] == 0


def test_eye_table_groups(renderer, soup, monkeypatch):
    """groups of 2 eye tables (TRACER_VIEW_GROUP): several closest-hit launches, the same bytes"""
    rs = renderer.upload(soup)
    renderer.trace_views(rs, _cams(EYES), W, H, rng_mode=1, seed=4)  # first frame: the shadow tables are built lazily
    whole = renderer.trace_views(rs, _cams(EYES), W, H, rng_mode=1, seed=4, debug=True)
    monkeypatch.setenv("TRACER_VIEW_GROUP", "2")
    for kw in (dict(rng_mode=1, seed=4), dict(rng_mode=0, seed=4, samples_per_pixel=4)):
        b = _batch_vs_singles(renderer, rs, EYES, **kw)
        if kw["rng_mode"] == 1:
            _same_frame(b, whole)
            # one eye table and one closest-hit launch more per extra group: 5 views in groups of 2 = 3 launches
            assert b.stats["kernel_launches"] == whole.stats["kernel_launches"] + 2
    fresh = renderer.upload(soup)  # a scene whose table buffer has never held more than 2 views
    _same_frame(renderer.trace_views(fresh, _cams(EYES), W, H, rng_mode=1, seed=4, debug=True), whole)


def test_device_output(renderer, soup):
    torch = pytest.importorskip("torch")
    rs = renderer.upload(soup)
    host = renderer.trace_views(rs, _cams(EYES), W, H, seed=8)
    buf = torch.zeros(len(EYES) * H * W * 3, dtype=torch.uint8, device="cuda")
    renderer.trace_views(rs, _cams(EYES), W, H, seed=8, out_device_ptr=buf.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(buf.cpu().numpy().reshape(host.rgb8.shape), host.rgb8)


def test_one_view_is_trace(renderer, soup):
    rs = renderer.upload(soup)
    cam = _cams(EYES[:1])
    for kw in (dict(rng_mode=0, seed=2), dict(rng_mode=1, seed=2), dict(rng_mode=0, seed=2, bvh=True)):
        renderer.trace(rs, cam[0], W, H, **kw)  # tables (and the tree) built before the compared frames
        a = renderer.trace_views(rs, cam, W, H, debug=True, **kw)
        b = renderer.trace(rs, cam[0], W, H, debug=True, **kw)
        _same_frame(a, b, 0)
        for key, val in b.stats.items():
            if not key.startswith("ms_"):
                assert a.stats[key] == val, key


def test_after_scene_update(renderer, soup):
    from esctp1raytracer_b200 import Scene

    rs = renderer.upload(soup)
    renderer.trace_views(rs, _cams(EYES), W, H, rng_mode=1, seed=6)  # tables built before the move
    g = 7  # move one geometry
    a, b = int(soup.geom_tri_offset[g]), int(soup.geom_tri_offset[g + 1])
    moved = soup.tri_verts.copy()
    moved[a:b] += np.float32([0.3, -0.2, 0.1])
    rs.update(tri_verts=moved[a:b], first_tri=a)
    batch = renderer.trace_views(rs, _cams(EYES), W, H, rng_mode=1, seed=6, debug=True)
    fresh = renderer.upload(Scene(soup.geom_tri_offset, moved, soup.geom_material, soup.light_geom, sphere_cr=soup.sphere_cr,
                                  sphere_material=soup.sphere_material))
    for v, cam in enumerate(_cams(EYES)):
        _same_frame(batch, renderer.trace(fresh, cam, W, H, rng_mode=1, seed=6, debug=True), v)


@pytest.mark.parametrize("name", golden_names())
def test_goldens_as_middle_view(renderer, name):
    """the reference's frame as view 1 of [other camera, golden camera, other camera]"""
    from esctp1raytracer_b200 import RNG_EXPLICIT, RNG_MT19937, Camera

    fs, fr = load_golden(name)
    w, h, L = fr["W"], fr["H"], len(fs.light_geom)
    eye = np.asarray(fr["eye"], np.float64)
    cams = [Camera.for_frame(eye + (0.4, 0.1, 0.2), fr["look"], w, h), Camera.for_frame(fr["eye"], fr["look"], w, h),
            Camera.for_frame(eye * 1.3 - (0.2, 0.0, 0.1), fr["look"], w, h)]
    rs = renderer.upload(to_scene(fs))

    def ppm(a):  # image index order (h*W+w) -> PPM row order
        return a.reshape(h, w, *a.shape[1:])[::-1].reshape(a.shape)

    fid = np.zeros((3, w * h * L), np.int32)
    fid[1] = np.asarray(fr["faceid"], np.int32).reshape(-1)
    for kw in (dict(rng_mode=RNG_MT19937, seed=fr["seed"]), dict(rng_mode=RNG_EXPLICIT, faceid=fid)):
        out = renderer.trace_views(rs, cams, w, h, debug=True, **kw)
        assert np.array_equal(out.tri[1], ppm(fr["tri"])), "hit ids differ"
        assert np.array_equal(bits(out.t[1]), bits(ppm(fr["t"]))) and np.array_equal(bits(out.v[1]), bits(ppm(fr["v"])))
        assert np.array_equal(bits(out.rgb[1]), bits(ppm(fr["rgb"]))), "float accumulator differs"
        assert np.array_equal(out.rgb8[1].reshape(-1, 3), np.asarray(fr["q"], np.uint8).reshape(-1, 3)), "PPM bytes differ"


def test_refusals(renderer, soup):
    from esctp1raytracer_b200 import RNG_EXPLICIT, _lib

    rs = renderer.upload(soup)
    cams = _cams(EYES[:2])
    carr = (_lib.CameraC * 2)(*[c.c for c in cams])
    out = np.zeros(2 * W * H * 3, np.uint8)
    dst = out.ctypes.data_as(C.c_void_p)

    def call(cam_ptr, n, **opt):
        o = _lib.RenderOpts()
        o.struct_size = C.sizeof(_lib.RenderOpts)
        for k, v in opt.items():
            setattr(o, k, v)
        return renderer.lib.tracer_cuda_render_views(rs.handle, cam_ptr, n, W, H, C.byref(o), dst)

    assert call(carr, 0) == -1 and call(None, 2) == -1
    assert call(carr, 2, bundle_cull=1) == -1
    assert call(carr, 2, band_rows=8, band_index=0, band_count=2) == -1
    many = (_lib.CameraC * 80000)(*([cams[0].c] * 80000))  # 80000 * 130 * 70 pixels: above the per-call limit
    assert call(many, 80000, rng_mode=0) == -1
    with pytest.raises(ValueError):
        renderer.trace_views(rs, cams, W, H, rng_mode=RNG_EXPLICIT, faceid=np.zeros((3, W * H * 4), np.int32))
    with pytest.raises(ValueError):
        renderer.trace_views(rs, [], W, H)
    with pytest.raises(ValueError):
        renderer.trace_views(rs, cams[0], W, H)
    with pytest.raises(ValueError):  # out: [V, H, W, 3]
        renderer.trace_views(rs, cams, W, H, out=np.zeros((2 * H, W, 3), np.uint8))
    after = renderer.trace_views(rs, cams, W, H, seed=3, debug=True)
    _same_frame(after, renderer.trace(rs, cams[1], W, H, seed=3, debug=True), 1)


def test_cli_eyes(soup, tmp_path):
    obj = tmp_path / "soup.obj"
    write_obj(soup, obj)
    cli = os.path.join(ROOT, "esctp1raytracer_b200", "tracer_cli.bin")
    eyes = ["0,1,3", "2.5,1.6,2", "-1.5,0.4,-2.8"]
    base = [cli, "-m", str(obj), "-l", "0,1,0", "-w", f"{W},{H}", "--seed", "7"]
    r = subprocess.run(base + sum((["--eye", e] for e in eyes), []) + ["-o", str(tmp_path / "views.ppm")], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    for i, e in enumerate(eyes):
        r = subprocess.run(base + ["-v", e, "-o", str(tmp_path / f"single{i}.ppm")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert (tmp_path / f"views_{i}.ppm").read_bytes() == (tmp_path / f"single{i}.ppm").read_bytes()
    for extra in (["-v", "0,1,3"], ["--cull"], ["--gpus", "2"]):
        r = subprocess.run(base + ["--eye", eyes[0]] + extra, capture_output=True, text=True)
        assert r.returncode != 0 and "--eye" in r.stderr
