"""The closest-hit sweep at 64 rays per thread (64-bit ray masks, 256 x 32 pixel tiles, its own launch bounds) on the
hot span rows: frames and every debug output bit-identical to 32 rays per thread and to the reference's frames, and
exhaustive mode — which also checks the hot loop's own per-triangle verdicts — finds no accept the filter would lose."""
import numpy as np
import pytest

from conftest import bits, golden_names, load_golden, to_flat, to_scene

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


def _no_misses(out):
    assert out.stats["filter_misses"] == 0 and out.stats["pipeline_errors"] == 0


@pytest.mark.parametrize("name", golden_names())
def test_r64_golden(renderer, name):
    """the reference's small frames, faceIDs replayed, at 64 rays per thread"""
    from esctp1raytracer_b200 import Camera, RNG_EXPLICIT

    fs, fr = load_golden(name)
    W, H = fr["W"], fr["H"]
    cam = Camera.for_frame(fr["eye"], fr["look"], W, H)
    rs = renderer.upload(to_scene(fs))
    out = renderer.trace(rs, cam, W, H, rng_mode=RNG_EXPLICIT, faceid=fr["faceid"], debug=True, rays_per_thread=64)
    assert np.array_equal(out.tri, _ppm(fr["tri"], W, H))
    assert np.array_equal(bits(out.t), bits(_ppm(fr["t"], W, H))) and np.array_equal(bits(out.v), bits(_ppm(fr["v"], W, H)))
    assert np.array_equal(bits(out.rgb), bits(_ppm(fr["rgb"], W, H)))
    assert np.array_equal(out.rgb8.reshape(-1, 3), np.asarray(fr["q"], np.uint8).reshape(-1, 3))
    ex = renderer.trace(rs, cam, W, H, rng_mode=RNG_EXPLICIT, faceid=fr["faceid"], debug=True, rays_per_thread=64, exhaustive_strict=True)
    _no_misses(ex)
    _same_frames(out, ex)


def _scenes():
    from esctp1raytracer_b200 import scenes
    from specular_scene import EYE, LOOK, specular_scene

    rng = np.random.default_rng(5)
    huge = scenes.soup_scene(200, 6, 2, seed=31, edge=(0.2, 1.5))  # big triangles all around the eye and the lights
    v = huge.tri_verts.reshape(-1, 3, 3).copy()
    for i in range(8, 40):  # axis-aligned edges
        v[i, 1] = v[i, 0] + np.array([rng.uniform(0.2, 2.0), 0.0, 0.0], np.float32)
        v[i, 2] = v[i, 0] + np.array([0.0, rng.uniform(0.2, 2.0), 0.0], np.float32)
    for i in range(40, 60):  # needles and zero-area triangles
        v[i, 1] = v[i, 0] + np.float32(1e-6) * rng.normal(size=3).astype(np.float32)
        v[i, 2] = v[i, 0] + (v[i, 1] - v[i, 0]) * np.float32(2.0) if i % 2 else v[i, 0]
    for i in range(60, 90):  # through the eye's plane
        v[i, 0, 2], v[i, 1, 2], v[i, 2, 2] = 2.0, 4.5, 3.0
    huge.tri_verts = np.ascontiguousarray(v, np.float32)
    return [
        ("soup", scenes.soup_scene(20000, 40, 4, seed=5), 300, 70, (0, 1, 3), (0, 1, 0)),  # ragged at both edges
        ("coplanar", scenes.coplanar_scene(), 120, 90, (0, 1, 2.9), (0, 1, 0)),
        ("huge", huge, 160, 90, (0, 1, 3), (0, 1, 0)),
        ("huge_oblique", huge, 97, 61, (0.3, 0.8, 0.5), (0.1, 1.0, -1.0)),
        ("specular", specular_scene(), 200, 150, EYE, LOOK),
    ]


@pytest.mark.parametrize("case", range(5))
def test_r64_equals_r32_and_the_oracle(renderer, restated, case):
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids

    name, s, W, H, eye, look = _scenes()[case]
    cam = Camera.for_frame(eye, look, W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, rays_per_thread=32)
    b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, rays_per_thread=64)
    _same_frames(a, b)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(3, W, H, s.faces_per_light))
    assert np.array_equal(b.tri, _ppm(o.tri, W, H)) and np.array_equal(b.occ_tri, _ppm(o.occ_tri, W, H)), name
    assert np.array_equal(bits(b.rgb), bits(_ppm(o.rgb, W, H))) and np.array_equal(b.rgb8.reshape(-1, 3), o.rgb8.reshape(-1, 3)), name
    ex = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, debug=True, rays_per_thread=64, exhaustive_strict=True)
    _no_misses(ex)
    _same_frames(b, ex)
    # bands (8-row bands, every third one) assembled into the frame
    frame = np.zeros_like(b.rgb8)
    for r in range(3):
        part = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, bands=(8, r, 3), rays_per_thread=64)
        frame[[pr for pr in range(H) if (pr // 8) % 3 == r]] = part.rgb8
    assert np.array_equal(frame, b.rgb8), name


def test_r64_random_bands_of_the_c4_frame(renderer):
    """random 8-row bands of the full C4 scene (1M triangles + 1k spheres, 3840 x 2160, 4 lights): the automatic choice
    (64 rays per thread) equals 32 rays per thread bit for bit, and exhaustive mode at 64 finds no miss"""
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    for band in np.random.default_rng(64).choice(H // 8, 2, replace=False):
        kw = dict(rng_mode=RNG_HASH, seed=seed, debug=True, bands=(8, int(band), H // 8))
        a = renderer.trace(rs, cam, W, H, rays_per_thread=32, **kw)
        b = renderer.trace(rs, cam, W, H, rays_per_thread=64, **kw)
        _same_frames(a, b)
        ex = renderer.trace(rs, cam, W, H, rays_per_thread=64, exhaustive_strict=True, **kw)
        _no_misses(ex)
        _same_frames(b, ex)
