"""GPU parity at the sizes BASELINE.json's configs name (VERDICT r1, "parity at real sizes").

C1/C2: CornellBox-Original at the reference's own 1024x768 (src/main.cpp:427, scripts/run.sh:28-30).
C3   : CornellBox-Sphere and CornellBox-Water at 1920x1080, in geometry order and in the
       flatten+sort order of src/simplify/flatten.cpp:50-82.
All five frames under tests/golden/full/ were rendered by the UNMODIFIED reference (scan_row through
oracle/ref_harness.cpp, tests/golden/make_golden.py big).  tri / q / faceid are stored whole; the float
arrays t / v / rgb as SHA-256 digests of their bytes (bit-exactness is what is claimed) plus every 97th pixel.
C4   : 1M triangles + 1k spheres at 3840x2160: 4096-pixel oracle subset, and the conservative filter checked
       exhaustively (every pair strict-tested) on random 8-row bands of the full-size scene.
C5   : 16 spp jittered primary rays (extension, parity unpinned: oracle = the restatement).
"""
import glob
import hashlib
import os

import numpy as np
import pytest
from conftest import GOLDEN, bits, to_flat

pytestmark = pytest.mark.gpu

FULL = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "full", "*.npz")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


def _load_full(name):
    from esctp1raytracer_b200 import Scene

    z = np.load(os.path.join(GOLDEN, "full", name + ".npz"))
    tn = z["tri_normals"]
    sc = Scene(z["geom_tri_offset"], z["tri_verts"], z["geom_material"], z["light_geom"],
               tri_normals=tn if len(tn) else None, geom_has_normals=z["geom_has_normals"])
    return sc, z


def _ppm(a, W, H):
    return a.reshape(H, W, *a.shape[1:])[::-1].reshape(a.shape)


def _image(a, W, H):
    """PPM row order -> image index order (h*W+w): the inverse of _ppm (a row flip is its own inverse)"""
    return _ppm(a, W, H)


def _check_against_reference(out, z, W, H):
    assert np.array_equal(out.tri, _ppm(z["tri"], W, H)), "hit ids differ from the reference's intersect()"
    stride = int(z["stride"])
    t, v, rgb = _image(out.t, W, H), _image(out.v, W, H), _image(out.rgb, W, H)
    # the strided samples first: they say WHERE a digest mismatch comes from
    assert np.array_equal(bits(t[::stride]), bits(z["t_s"])), "closest-hit t differs"
    assert np.array_equal(bits(v[::stride]), bits(z["v_s"])), "closest-hit v differs"
    assert sha(t) == str(z["sha_t"]) and sha(v) == str(z["sha_v"])
    # specular frames (C3: ks != 0) included: the device's powf is glibc's own (strict::powf_glibc)
    assert np.array_equal(bits(rgb[::stride]), bits(z["rgb_s"])), "float accumulator differs"
    assert sha(rgb) == str(z["sha_rgb"]), "float accumulator differs from scan_row's"
    assert np.array_equal(out.rgb8.reshape(-1, 3), z["q"].reshape(-1, 3)), "PPM bytes differ"


@pytest.mark.parametrize("name", FULL)
def test_reference_frame_at_configured_size(renderer, name):
    """seed only: the library's std::mt19937 replay + the CUDA path reproduce the reference's seeded frame"""
    from esctp1raytracer_b200 import RNG_EXPLICIT, RNG_MT19937, Camera

    sc, z = _load_full(name)
    W, H = int(z["W"]), int(z["H"])
    cam = Camera.for_frame(z["eye"], z["look"], W, H)
    assert np.array_equal(cam.as_array(), z["cam"])
    rs = renderer.upload(sc)
    out = renderer.trace(rs, cam, W, H, rng_mode=RNG_MT19937, seed=int(z["seed"]), debug=True)
    _check_against_reference(out, z, W, H)
    assert out.stats["tests_primary"] == W * H * sc.n_tris
    # explicit faceIDs (the replay the harness recorded) and the optional bundle-cull mode give the same bytes
    fid = z["faceid"].astype(np.int32)
    out2 = renderer.trace(rs, cam, W, H, rng_mode=RNG_EXPLICIT, faceid=fid, bundle_cull=True)
    assert np.array_equal(out2.rgb8, out.rgb8)


def test_sorted_order_changes_ids_only_where_the_order_matters(renderer):
    """C3 'full vs simplify-reduced': same geometry, different iteration order => the images may differ only through
    ties / first-occluder order; mapped back through (geom_id, prim_id) the closest hits name the same triangles
    wherever t is not tied."""
    if "c3_sphere_1080p" not in FULL or "c3_sphere_1080p_sorted" not in FULL:
        pytest.skip("fixtures missing")
    base, zb = _load_full("c3_sphere_1080p")
    srt, zs = _load_full("c3_sphere_1080p_sorted")
    origin = zs["origin"]
    tb, ts = zb["tri"], zs["tri"]
    assert ((tb >= 0) == (ts >= 0)).all()
    hit = tb >= 0
    back = base.geom_tri_offset[origin[ts[hit], 0]] + origin[ts[hit], 1]
    differ = back != tb[hit]
    assert differ.mean() < 1e-3  # ties only


def test_c4_full_size_oracle_subset_and_filter_soundness(renderer, restated):
    """BASELINE.json configs[3] at full size.  (1) 4096 random pixels (SURVEY 8d-C4) against the restatement, bit for
    bit: ids, t, per-light occluders, float accumulator, bytes.  (2) The default and bundle-cull modes read the SAME
    filter tables, so comparing them cannot see a too-tight margin; exhaustive_strict can: every (ray, triangle) pair
    of four random 8-row bands of the full-size scene is strict-tested and accepts the filter would have lost are
    counted — 0 for both sweeps — and the band's bytes equal the default mode's."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, hash_faceids, scenes

    W, H, seed = 3840, 2160, 42
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True)
    assert a.stats["n_primary_rays"] == W * H and a.stats["tests_primary"] == W * H * 1_000_000
    assert (a.tri >= 0).sum() * 4 == a.stats["n_shadow_rays"]
    fid = hash_faceids(seed, W, H, s.faces_per_light)
    idx = np.random.default_rng(1).choice(W * H, 4096, replace=False)
    ph, pw = idx // W, idx % W
    restated.set_simd(True)  # the AVX2 form is pinned bit-identical to the scalar loops (test_oracle_pin.py)
    try:
        o = restated.render_pixels(to_flat(s), cam.as_array(), W, H, pw, ph, fid[idx], n_threads=os.cpu_count() or 1)
    finally:
        restated.set_simd(False)
    k = (H - 1 - ph) * W + pw
    assert np.array_equal(a.tri[k], o.tri)
    assert np.array_equal(bits(a.t[k]), bits(o.t))
    assert np.array_equal(a.occ_tri[k], o.occ_tri)
    assert np.array_equal(bits(a.rgb[k]), bits(o.rgb))
    assert np.array_equal(a.rgb8.reshape(-1, 3)[k], o.rgb8)
    n_bands = H // 8
    for r in np.random.default_rng(2).choice(n_bands, 4, replace=False):
        b = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=seed, debug=True, bands=(8, int(r), n_bands),
                           exhaustive_strict=True)
        assert b.stats["filter_misses"] == 0 and b.stats["pipeline_errors"] == 0
        rows = slice(int(r) * 8, int(r) * 8 + 8)
        assert np.array_equal(b.rgb8, a.rgb8[rows])
        assert np.array_equal(b.tri, a.tri.reshape(H, W)[rows].reshape(-1))
        assert np.array_equal(b.occ_tri, a.occ_tri.reshape(H, W, 4)[rows].reshape(-1, 4))


def test_16spp_jittered_parity(renderer, restated):
    """BASELINE.json configs[4]'s sampling (16 spp stratified jitter; extension, parity unpinned): GPU == restatement."""
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    s = scenes.soup_scene(20000, 40, 1, seed=8)
    W, H = 256, 144
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    rs = renderer.upload(s)
    out = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, samples_per_pixel=16, debug=True)
    rgb, rgb8 = restated.render_spp(to_flat(s), cam.as_array(), W, H, 3, 4)
    assert np.array_equal(bits(out.rgb), bits(_ppm(rgb, W, H)))
    assert np.array_equal(out.rgb8, rgb8)
    cull = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=3, samples_per_pixel=16, bundle_cull=True)
    assert np.array_equal(cull.rgb8, rgb8)
