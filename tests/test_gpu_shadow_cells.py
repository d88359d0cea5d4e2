"""Shadow sweeps with the rays of each group ordered in serpentine p-sorted stripes of the q-sorted list and decided per
thread by the mean-q segment verdict (sweep.cuh: segment_pass after hot_terms_qbar): every debug output (hit ids/t/v,
per-light occluder ids, float accumulator, u8 frame) equals the restatement oracle and bundle-cull mode, for stripe lengths
of one entry (plain q order), 4096 entries (one ray block) and the default, with 2, 32 and 64 shadow chunks, in 8-row band
shares (the part-filled 16/8/4/2-ray instantiations), seeded faceIDs, a crop window, and in exhaustive mode
(filter_misses == 0 and pipeline_errors == 0)."""
import os

import numpy as np
import pytest

from conftest import bits, to_flat
from test_gpu_shadow_lanes import _cases, _no_misses, _ppm, _same_frames

pytestmark = pytest.mark.gpu

STRIPES = (None, "1", "4096")


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


@pytest.fixture
def stripe():
    old = os.environ.get("TRACER_SHADOW_STRIPE")

    def set_len(v):
        if v is None:
            os.environ.pop("TRACER_SHADOW_STRIPE", None)
        else:
            os.environ["TRACER_SHADOW_STRIPE"] = v

    yield set_len
    set_len(old)


@pytest.mark.parametrize("case", [0, 1, 6])  # soup with 4 lights, the hot-row soup, edge-on triangles
def test_cells_equal_the_oracle_and_bundle_cull(renderer, restated, stripe, case):
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids

    name, s, W, H, eye, look = _cases()[case]
    cam = Camera.for_frame(eye, look, W, H)
    rs = renderer.upload(s)
    kw = dict(rng_mode=RNG_HASH, seed=5, debug=True)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(5, W, H, s.faces_per_light))
    cull = renderer.trace(rs, cam, W, H, bundle_cull=True, **kw)
    for L in STRIPES:
        stripe(L)
        a = renderer.trace(rs, cam, W, H, **kw)
        _no_misses(a)
        assert np.array_equal(a.tri, _ppm(o.tri, W, H)) and np.array_equal(a.occ_tri, _ppm(o.occ_tri, W, H)), (name, L)
        assert np.array_equal(bits(a.t), bits(_ppm(o.t, W, H))) and np.array_equal(bits(a.v), bits(_ppm(o.v, W, H))), (name, L)
        assert np.array_equal(bits(a.rgb), bits(_ppm(o.rgb, W, H))) and np.array_equal(a.rgb8.reshape(-1, 3), o.rgb8.reshape(-1, 3)), (name, L)
        _same_frames(a, cull)
        for chunks in (2, 32, 64):
            ex = renderer.trace(rs, cam, W, H, shadow_chunks=chunks, exhaustive_strict=True, **kw)
            _no_misses(ex)
            _same_frames(a, ex)
        for ex in (False, True):  # 8-row band shares: few rays per group, part-filled blocks
            frame = np.zeros_like(a.rgb8)
            for r in range(3):
                part = renderer.trace(rs, cam, W, H, bands=(8, r, 3), shadow_chunks=32, exhaustive_strict=ex, **kw)
                _no_misses(part)
                frame[[pr for pr in range(H) if (pr // 8) % 3 == r]] = part.rgb8
            assert np.array_equal(frame, a.rgb8), (name, L, ex)


def test_cells_seeded_faceids_and_crop(renderer, stripe):
    from esctp1raytracer_b200 import RNG_MT19937, Camera

    name, s, W, H, eye, look = _cases()[6]
    cam = Camera.for_frame(eye, look, W, H)
    rs = renderer.upload(s)
    kw = dict(rng_mode=RNG_MT19937, seed=7, debug=True)
    cull = renderer.trace(rs, cam, W, H, bundle_cull=True, **kw)
    for L in STRIPES:
        stripe(L)
        a = renderer.trace(rs, cam, W, H, exhaustive_strict=True, **kw)
        _no_misses(a)
        _same_frames(a, cull)
        x, y, w, h = 37, 51, 120, 90
        c = renderer.trace(rs, cam, W, H, crop=(x, y, w, h), **kw)
        assert np.array_equal(c.rgb8, a.rgb8[y:y + h, x:x + w]), (name, L)
