"""The warp-wide candidate pass (sweep.cuh: flagged pairs queued per warp and drained one per lane) and the shadow sweep
at 32 rays per thread: every debug output (hit ids/t/v, per-light occluder ids, float accumulator, u8 frame) equals the
restatement oracle and bundle-cull mode, with 2 and 64 shadow chunks, in 8-row band shares (the small ray blocks run the
16/8/4/2-ray instantiations) and in exhaustive mode, which queues every pair, so each batch overflows the queue and
drains it in rounds."""
import numpy as np
import pytest

from conftest import bits, to_flat
from test_gpu_hot_rows import _scenes as _hot_row_scenes

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


def _edge_on_scene():
    """a 4-light soup plus triangles whose planes pass through a light vertex: seen from that vertex each one is a
    segment, and the shadow rays around it flag the same triangle across many lanes of a warp"""
    from esctp1raytracer_b200 import scenes

    s = scenes.soup_scene(3000, 12, 4, seed=17, edge=(0.02, 0.08))
    rng = np.random.default_rng(17)
    v = s.tri_verts.reshape(-1, 3, 3).copy()
    lights = v[4:12].reshape(-1, 3)  # the 4 quad lights' vertices
    for i in range(12, 1200):
        L = lights[rng.integers(len(lights))].astype(np.float64)
        c = rng.uniform([-0.9, 0.2, -0.9], [0.9, 1.7, 0.9])
        d = (c - L) / np.linalg.norm(c - L)
        e = np.cross(d, rng.normal(size=3))
        e /= np.linalg.norm(e)
        a, b = rng.uniform(0.05, 0.3, size=2)
        v[i] = np.array([c, c + a * d + 0.5 * b * e, c - a * d + b * e], np.float32)
    s.tri_verts = np.ascontiguousarray(v, np.float32)
    return s


def _cases():
    from esctp1raytracer_b200 import scenes

    hot = {c[0]: c for c in _hot_row_scenes()}
    return [
        ("soup_4_lights", scenes.soup_scene(2000, 10, 4, seed=9, edge=(0.03, 0.1)), 480, 270, (0, 1, 3), (0, 1, 0)),
        hot["soup"], hot["coplanar"], hot["huge"], hot["huge_oblique"], hot["specular"],
        ("edge_on", _edge_on_scene(), 400, 240, (0, 1, 3), (0, 1, 0)),
    ]


@pytest.mark.parametrize("case", range(7))
def test_shadow_lanes_equal_the_oracle_and_bundle_cull(renderer, restated, case):
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids

    name, s, W, H, eye, look = _cases()[case]
    cam = Camera.for_frame(eye, look, W, H)
    rs = renderer.upload(s)
    kw = dict(rng_mode=RNG_HASH, seed=3, debug=True)
    a = renderer.trace(rs, cam, W, H, **kw)
    _no_misses(a)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(3, W, H, s.faces_per_light))
    assert np.array_equal(a.tri, _ppm(o.tri, W, H)) and np.array_equal(a.occ_tri, _ppm(o.occ_tri, W, H)), name
    assert np.array_equal(bits(a.t), bits(_ppm(o.t, W, H))) and np.array_equal(bits(a.v), bits(_ppm(o.v, W, H))), name
    assert np.array_equal(bits(a.rgb), bits(_ppm(o.rgb, W, H))) and np.array_equal(a.rgb8.reshape(-1, 3), o.rgb8.reshape(-1, 3)), name
    _same_frames(a, renderer.trace(rs, cam, W, H, bundle_cull=True, **kw))
    for chunks in (2, 64):
        _same_frames(a, renderer.trace(rs, cam, W, H, shadow_chunks=chunks, **kw))
        ex = renderer.trace(rs, cam, W, H, shadow_chunks=chunks, exhaustive_strict=True, **kw)
        _no_misses(ex)
        _same_frames(a, ex)
    # 8-row band shares (every third band): few rays per light vertex and cube face, so the part-filled blocks run
    for chunks in (2, 64):
        for ex in (False, True):
            frame = np.zeros_like(a.rgb8)
            for r in range(3):
                part = renderer.trace(rs, cam, W, H, bands=(8, r, 3), shadow_chunks=chunks, exhaustive_strict=ex, **kw)
                _no_misses(part)
                frame[[pr for pr in range(H) if (pr // 8) % 3 == r]] = part.rgb8
            assert np.array_equal(frame, a.rgb8), (name, chunks, ex)
