"""CPU side of the full-size fixtures (tests/golden/full, rendered by the UNMODIFIED reference at the sizes
BASELINE.json's configs name): the flatten+sort host helper, and the restatement pinned against the reference's
frames at 1024x768 / 1920x1080 (not only at thumbnail size)."""
import glob
import hashlib
import os

import numpy as np
import pytest
from conftest import GOLDEN, bits

FULL = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "full", "*.npz")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _load_full(name):
    from esctp1raytracer_b200 import Scene

    z = np.load(os.path.join(GOLDEN, "full", name + ".npz"))
    tn = z["tri_normals"]
    sc = Scene(z["geom_tri_offset"], z["tri_verts"], z["geom_material"], z["light_geom"],
               tri_normals=tn if len(tn) else None, geom_has_normals=z["geom_has_normals"])
    return sc, z


def test_fixtures_present():
    assert {"c1_cornell_original_1024x768", "c3_sphere_1080p", "c3_sphere_1080p_sorted", "c3_water_1080p",
            "c3_water_1080p_sorted"} <= set(FULL)


@pytest.mark.parametrize("name", [n for n in FULL if n.endswith("_sorted")])
def test_flatten_sorted_helper_builds_the_sorted_scene(name):
    """tracer_scene_flatten_sorted (src/simplify/flatten.cpp:50-82, comparator :20-27) applied to the geometry-order
    scene == the scene the reference rendered the sorted golden from"""
    base, _ = _load_full(name[: -len("_sorted")])
    want, z = _load_full(name)
    got, og, op = base.flatten_sorted()
    assert np.array_equal(got.geom_tri_offset, want.geom_tri_offset)
    assert np.array_equal(bits(got.tri_verts), bits(want.tri_verts))
    assert np.array_equal(got.light_geom, want.light_geom)
    assert np.array_equal(bits(got.geom_material), bits(want.geom_material))
    assert np.array_equal(np.stack([og, op], 1), z["origin"])
    n = base.n_tris
    x = got.tri_verts[:n, 0, 0]
    assert (np.diff(x) >= 0).all(), "not sorted by vertices[0].x (flatten.cpp:20-27)"
    # stable: equal keys keep (geometry, face) order; every input triangle appears exactly once in the sorted part
    flat_id = base.geom_tri_offset[og[:n]] + op[:n]
    assert sorted(flat_id.tolist()) == list(range(n))
    same = np.diff(x) == 0
    assert (np.diff(flat_id)[same] > 0).all()
    # the light geometries follow, once more, in their original face order (light.vertex[faceID], main.cpp:749)
    for lg_new, lg_old in zip(got.light_geom, base.light_geom):
        a = got.tri_verts[got.geom_tri_offset[lg_new]:got.geom_tri_offset[lg_new + 1]]
        b = base.tri_verts[base.geom_tri_offset[lg_old]:base.geom_tri_offset[lg_old + 1]]
        assert np.array_equal(bits(a), bits(b))


def test_flatten_sorted_rejects_bad_input():
    from esctp1raytracer_b200 import Scene, TracerError

    sc = Scene(np.array([0, 1], np.int32), np.zeros((1, 3, 3), np.float32), np.zeros((1, 13), np.float32), np.array([3], np.int32))
    with pytest.raises(TracerError):
        sc.flatten_sorted()


@pytest.mark.parametrize("name", FULL)
def test_restatement_equals_reference_at_configured_size(restated, name):
    """oracle/restated.c (AVX2 form, itself pinned bit-identical to the scalar loops) against the reference's own
    frame at the configured resolution: ids, t, v, float accumulator (digests) and PPM bytes."""
    from conftest import to_flat

    sc, z = _load_full(name)
    W, H = int(z["W"]), int(z["H"])
    if not restated.set_simd(True):
        pytest.skip("no AVX2 on this host: the scalar restatement needs minutes at this size")
    try:
        o = restated.render(to_flat(sc), z["cam"], W, H, faceid=z["faceid"].astype(np.int32))
    finally:
        restated.set_simd(False)
    assert np.array_equal(o.tri, z["tri"])
    assert sha(o.t) == str(z["sha_t"]) and sha(o.v) == str(z["sha_v"])
    assert sha(o.rgb) == str(z["sha_rgb"])  # specular frames too: libm powf is what the reference called
    assert np.array_equal(o.rgb8, z["q"])
