"""Specular shading on the device, bit for bit: the shading's powf is strict::powf_glibc (csrc/strict_math.cuh), glibc's
own powf (tests/test_powf_glibc.py pins its host build to libm).

1. The device build of the port against the host build, over every float x in [0, 1.0001] for every Ns of the
   reference's scenes and over random (x, y) pairs: nvcc must have compiled it to the same operations.
2. The reference's own specular frames (ks != 0) at thumbnail size, faceIDs replayed and from the seed.
3. A specular-dominated scene (tests/specular_scene.py: high ks, low kd, ten different Ns, 4 lights) in the default
   mode, the bundle-cull mode, row bands and 2x2 samples per pixel, against the restatement.
"""
import ctypes as C

import numpy as np
import pytest
from conftest import bits, load_golden, to_flat, to_scene
from specular_scene import EYE, LOOK, NS, SEED, specular_scene
from test_powf_glibc import GOLDEN_NS, ONE_PLUS, random_pairs

pytestmark = pytest.mark.gpu

F32 = np.float32
F32P = C.POINTER(C.c_float)
MAX_REP = 8
CHUNK = 1 << 26  # x values per device call (256 MB of results)


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


@pytest.fixture(scope="module")
def host_port(tmp_path_factory):
    import os
    import subprocess

    from conftest import ROOT

    so = tmp_path_factory.mktemp("powf_host") / "libstrict_host.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-I/usr/local/cuda/include",
                        os.path.join(ROOT, "tests", "strict_host_shim.cpp"), "-o", str(so)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(str(so))
    lib.strict_host_powf_compare_range.restype = C.c_int64
    lib.strict_host_powf_compare_range.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, F32P, C.c_int, F32P, C.c_int]
    lib.strict_host_powf_compare_pairs.restype = C.c_int64
    lib.strict_host_powf_compare_pairs.argtypes = [C.c_int64, F32P, F32P, F32P, C.c_int, F32P, C.c_int]
    return lib


@pytest.fixture(scope="module")
def device_port(renderer):
    from esctp1raytracer_b200 import _lib

    lib = _lib.load()
    lib.tracer__device_powf.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, F32P]
    lib.tracer__device_powf_pairs.argtypes = [C.c_int64, F32P, F32P, F32P]
    return lib


def _n_threads():
    import os

    return os.cpu_count() or 1


def _report(count, rep, what):
    rows = [tuple(float(v) for v in rep[4 * k:4 * k + 4]) for k in range(min(count, MAX_REP))]
    return f"{what}: {count} device results differ from the host port; first (x, y, device, host): {rows}"


@pytest.mark.parametrize("ns", GOLDEN_NS)
def test_device_port_equals_host_port_for_every_x_in_0_to_1(device_port, host_port, ns):
    from esctp1raytracer_b200._lib import check

    got = np.zeros(CHUNK, F32)
    rep = np.zeros(4 * MAX_REP, F32)
    total = 0
    for lo in range(0, ONE_PLUS + 1, CHUNK):
        hi = min(lo + CHUNK - 1, ONE_PLUS)
        check(device_port.tracer__device_powf(lo, hi, 1, ns, got.ctypes.data_as(F32P)))
        n = host_port.strict_host_powf_compare_range(lo, hi, 1, ns, got.ctypes.data_as(F32P), _n_threads(),
                                                     rep.ctypes.data_as(F32P), MAX_REP)
        assert n == 0, _report(n, rep, f"y = {ns}, x bits [{lo:#x}, {hi:#x}]")
        total += hi - lo + 1
    assert total == ONE_PLUS + 1


def test_device_port_equals_host_port_for_random_pairs(device_port, host_port):
    from esctp1raytracer_b200._lib import check

    x, y = random_pairs(10_000_000, 7)
    got = np.zeros_like(x)
    check(device_port.tracer__device_powf_pairs(len(x), x.ctypes.data_as(F32P), y.ctypes.data_as(F32P), got.ctypes.data_as(F32P)))
    rep = np.zeros(4 * MAX_REP, F32)
    n = host_port.strict_host_powf_compare_pairs(len(x), x.ctypes.data_as(F32P), y.ctypes.data_as(F32P), got.ctypes.data_as(F32P),
                                                 _n_threads(), rep.ctypes.data_as(F32P), MAX_REP)
    assert n == 0, _report(n, rep, "random pairs")


def _ppm(a, W, H):
    """image index order (h*W+w) <-> PPM row order (row 0 = h=H-1)"""
    return a.reshape(H, W, *a.shape[1:])[::-1].reshape(a.shape)


def _check(out, W, H, o):
    """every debug output of the device frame == the restatement's (o: image index order)"""
    assert out.stats["pipeline_errors"] == 0 and out.stats["filter_misses"] == 0
    assert np.array_equal(out.tri, _ppm(o.tri, W, H)), "hit ids differ"
    assert np.array_equal(bits(out.t), bits(_ppm(o.t, W, H))), "closest-hit t differs"
    assert np.array_equal(bits(out.v), bits(_ppm(o.v, W, H))), "closest-hit v differs"
    assert np.array_equal(out.occ_tri, _ppm(o.occ_tri, W, H)), "shadow decisions differ"
    assert np.array_equal(bits(out.rgb), bits(_ppm(o.rgb, W, H))), "float accumulator differs"
    assert np.array_equal(out.rgb8.reshape(-1, 3), o.rgb8.reshape(-1, 3)), "PPM bytes differ"


@pytest.mark.parametrize("name", ["cornell_sphere", "cornell_water", "cornell_box_ks"])
def test_reference_specular_frames(renderer, name):
    """the reference's own frames with ks != 0: float accumulator and bytes, faceIDs replayed and from the seed"""
    from esctp1raytracer_b200 import RNG_EXPLICIT, RNG_MT19937, Camera

    fs, fr = load_golden(name)
    assert fs.geom_material[:, 6:9].any()
    W, H = fr["W"], fr["H"]
    cam = Camera.for_frame(fr["eye"], fr["look"], W, H)
    rs = renderer.upload(to_scene(fs))
    for kw in (dict(rng_mode=RNG_EXPLICIT, faceid=fr["faceid"]), dict(rng_mode=RNG_MT19937, seed=fr["seed"])):
        out = renderer.trace(rs, cam, W, H, debug=True, **kw)
        assert out.stats["pipeline_errors"] == 0
        assert np.array_equal(out.tri, _ppm(fr["tri"], W, H))
        assert np.array_equal(bits(out.rgb), bits(_ppm(fr["rgb"], W, H))), "float accumulator differs"
        assert np.array_equal(out.rgb8.reshape(-1, 3), np.asarray(fr["q"], np.uint8).reshape(-1, 3)), "PPM bytes differ"


@pytest.fixture(scope="module")
def specular(renderer, restated):
    from esctp1raytracer_b200 import Camera, hash_faceids

    s = specular_scene()
    W, H = 320, 240
    cam = Camera.for_frame(EYE, LOOK, W, H)
    o = restated.render(to_flat(s), cam.as_array(), W, H, faceid=hash_faceids(SEED, W, H, s.faces_per_light))
    return s, renderer.upload(s), cam, W, H, o


@pytest.mark.parametrize("bundle_cull", [False, True], ids=["default", "bundle_cull"])
def test_specular_scene(renderer, specular, bundle_cull):
    from esctp1raytracer_b200 import RNG_HASH

    s, rs, cam, W, H, o = specular
    out = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=SEED, debug=True, bundle_cull=bundle_cull)
    _check(out, W, H, o)
    # the scene is what it claims: many pixels lit by several lights, surfaces of every Ns in view
    assert ((o.occ_tri == -1).sum(axis=1) >= 2).sum() > W * H // 4
    g = np.searchsorted(s.geom_tri_offset, o.tri[(o.tri >= 0) & (o.tri < s.n_tris)], "right") - 1
    ns_seen = {float(s.geom_material[k, 12]) for k in np.unique(g) if k not in s.light_geom}
    ns_seen |= {float(s.sphere_material[i - s.n_tris, 12]) for i in np.unique(o.tri[o.tri >= s.n_tris])}
    assert ns_seen == {float(F32(x)) for x in NS}, ns_seen


def test_specular_scene_in_bands(renderer, specular):
    """interleaved 8-row bands (what each rank of a multi-GPU frame renders), put back together"""
    from esctp1raytracer_b200 import RNG_HASH

    s, rs, cam, W, H, o = specular
    B, n = 8, 3
    tri = np.zeros(W * H, np.int32).reshape(H, W)
    t, v, rgb = np.zeros((H, W), F32), np.zeros((H, W), F32), np.zeros((H, W, 3), F32)
    occ = np.zeros((H, W, s.n_lights), np.int32)
    rgb8 = np.zeros((H, W, 3), np.uint8)
    for r in range(n):
        part = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=SEED, debug=True, bands=(B, r, n))
        assert part.stats["pipeline_errors"] == 0
        rows = [pr for pr in range(H) if (pr // B) % n == r]
        tri[rows] = part.tri.reshape(-1, W)
        t[rows], v[rows] = part.t.reshape(-1, W), part.v.reshape(-1, W)
        rgb[rows] = part.rgb.reshape(-1, W, 3)
        occ[rows] = part.occ_tri.reshape(-1, W, s.n_lights)
        rgb8[rows] = part.rgb8
    assert np.array_equal(tri.reshape(-1), _ppm(o.tri, W, H))
    assert np.array_equal(bits(t).reshape(-1), bits(_ppm(o.t, W, H))) and np.array_equal(bits(v).reshape(-1), bits(_ppm(o.v, W, H)))
    assert np.array_equal(occ.reshape(-1, s.n_lights), _ppm(o.occ_tri, W, H))
    assert np.array_equal(bits(rgb).reshape(-1, 3), bits(_ppm(o.rgb, W, H))), "float accumulator differs"
    assert np.array_equal(rgb8, o.rgb8)


def test_specular_scene_2x2_samples_per_pixel(renderer, restated, specular):
    from esctp1raytracer_b200 import RNG_HASH

    s, rs, cam, W, H, _ = specular
    rgb, rgb8 = restated.render_spp(to_flat(s), cam.as_array(), W, H, SEED, 2)
    for bundle_cull in (False, True):
        out = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=SEED, samples_per_pixel=4, debug=True, bundle_cull=bundle_cull)
        assert out.stats["pipeline_errors"] == 0
        assert np.array_equal(bits(out.rgb), bits(_ppm(rgb, W, H))), "float accumulator differs"
        assert np.array_equal(out.rgb8, rgb8)
