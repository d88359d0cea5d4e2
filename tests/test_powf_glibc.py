"""strict::powf_glibc (csrc/strict_math.cuh), the shading's powf, against the host's libm powf, bit for bit.

The reference shades with libm powf(dot(N,H), Ns) (main.cpp:783).  glibc's powf is not correctly rounded, so the device
reproduces glibc's own algorithm, in the variant x86-64 hosts with FMA + AVX2 select.  Here the port is compiled for
the host (tests/strict_host_shim.cpp) and compared with libm over every float x in [0, 1.0001] (the range dot(N,H)
takes) for every Ns the reference's scenes use, over every 5th float for edge exponents, and over random (x, y) pairs
that reach the special cases.  The comparison loops run in C on all cores; Python only reads mismatch counts.

The same harness run on the formula the shading used before, (float)pow((double)x, (double)y), reports mismatches,
and the reference's own C3 frames and the specular scene of tests/specular_scene.py render differently with it: the
comparison is not vacuous, and the frames would catch a regression.
"""
import ctypes as C
import glob
import hashlib
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
from conftest import GOLDEN, ROOT, to_flat

CUDA_INC = "/usr/local/cuda/include"
F32 = np.float32
F32P = C.POINTER(C.c_float)
N_THREADS = os.cpu_count() or 1
MAX_REP = 8
PORT, OLD_FORMULA = 0, 1


def fbits(x):
    return int(np.array(x, F32).view(np.uint32))


ONE_PLUS = fbits(1.0001)  # top of the exhaustive range of x
# every Ns of the reference's scenes (tests/golden, tests/golden/full) and the synthetic soups' 10
GOLDEN_NS = sorted({float(n) for p in glob.glob(os.path.join(GOLDEN, "*.npz")) + glob.glob(os.path.join(GOLDEN, "full", "*.npz"))
                    for n in np.load(p)["geom_material"][:, 12]} | {10.0})
EDGE_Y = [0.0, float(np.array(1, np.uint32).view(F32)), 0.5, 1.0, 2.0, 3.0, 7.3, 64.0, 127.99, 4096.0, 1e6, -1.0, -10.0,
          math.inf, -math.inf, math.nan]


def libc_version():
    try:
        f = C.CDLL(None).gnu_get_libc_version
        f.restype = C.c_char_p
        return "glibc " + f().decode()
    except (AttributeError, OSError):
        return "not glibc"


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not shutil.which("g++") or not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA headers")
    so = tmp_path_factory.mktemp("powf") / "libstrict_host.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-I" + CUDA_INC,
                        os.path.join(ROOT, "tests", "strict_host_shim.cpp"), "-o", str(so)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(str(so))
    lib.strict_host_powf_check_range.restype = C.c_int64
    lib.strict_host_powf_check_range.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_int, C.c_int, F32P, C.c_int]
    lib.strict_host_powf_check_pairs.restype = C.c_int64
    lib.strict_host_powf_check_pairs.argtypes = [C.c_int64, F32P, F32P, C.c_int, C.c_int, F32P, C.c_int]
    lib.strict_host_powf_tables.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    lib.strict_host_powf_tables.restype = None
    if not lib.strict_host_has_fma_avx2() or libc_version() == "not glibc":
        pytest.skip(f"libm here is {libc_version()} on a CPU without FMA + AVX2: its powf is not the variant the port "
                    "reproduces (glibc's FMA variant, which x86-64 hosts with FMA + AVX2 select)")
    return lib


def _report(count, rep, what):
    rows = [tuple(float(v) for v in rep[4 * k:4 * k + 4]) for k in range(min(count, MAX_REP))]
    return (f"{what}: {count} mismatches against libm powf ({libc_version()}); first (x, y, got, want): "
            + ", ".join(f"({x!r}, {y!r}, {g!r}, {w!r})" for x, y, g, w in rows))


def check_range(lib, lo, hi, stride, y, impl=PORT):
    rep = np.zeros(4 * MAX_REP, F32)
    n = lib.strict_host_powf_check_range(lo, hi, stride, y, impl, N_THREADS, rep.ctypes.data_as(F32P), MAX_REP)
    return n, rep


def random_pairs(n, seed):
    """(x, y) over the whole float range, weighted towards the special cases: negative x with integer and non-integer y,
    +-0, +-inf, NaN (quiet and signaling), subnormals, exponents near the overflow / underflow thresholds"""
    rng = np.random.default_rng(seed)
    xb = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)  # any bit pattern
    yb = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    x, y = xb.view(F32), yb.view(F32)
    k = rng.integers(0, 8, n)
    # moderate |x| and y, so that x^y stays finite and non-zero
    m = k == 1
    x[m] = (rng.uniform(-4, 4, m.sum()) * 2.0 ** rng.integers(-20, 20, m.sum())).astype(F32)
    y[m] = rng.uniform(-30, 30, m.sum()).astype(F32)
    # negative x, integer y (odd and even, both signs, up to and beyond 2^24)
    m = k == 2
    x[m] = -np.abs(x[m])
    y[m] = (rng.integers(-2 ** 25, 2 ** 25, m.sum()) >> rng.integers(0, 25, m.sum())).astype(F32)
    # subnormal x
    m = k == 3
    x[m] = rng.integers(1, 1 << 23, m.sum(), dtype=np.uint32).view(F32) * rng.choice(np.array([1, -1], F32), m.sum())
    y[m] = rng.uniform(-2, 2, m.sum()).astype(F32)
    # special values on either side
    sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, -1.0, 2.0 ** -149, -(2.0 ** -149), 2.0 ** -126,
                   np.array(0x7fa00000, np.uint32).view(F32), np.array(0xffc00001, np.uint32).view(F32)], F32)
    m = k == 4
    x[m] = rng.choice(sp, m.sum())
    m = k == 5
    y[m] = rng.choice(np.concatenate([sp, np.array([0.5, -0.5, 3.0, -3.0, 2.0 ** 30, -(2.0 ** 30)], F32)]), m.sum())
    # y*log2(x) near the overflow (128) and underflow (-126 .. -150) thresholds
    m = k == 6
    x[m] = rng.uniform(0.5, 2.0, m.sum()).astype(F32)
    t = rng.uniform(-151, 129, m.sum())
    with np.errstate(divide="ignore"):
        y[m] = (t / np.log2(x[m].astype(np.float64))).astype(F32)
    return np.ascontiguousarray(x), np.ascontiguousarray(y)


def test_tables_match_their_formulas(shim):
    """exp2 table: entry i = asuint64(2^(i/32)) - (i << 52)/32; log2 table: logc = log2(c) for c = 1/invc, and 1/invc lies
    near the subinterval the index selects"""
    lg = np.zeros(32, np.float64)
    ex = np.zeros(32, np.uint64)
    shim.strict_host_powf_tables(lg.ctypes.data_as(C.POINTER(C.c_double)), ex.ctypes.data_as(C.POINTER(C.c_uint64)))
    for i in range(32):
        want = int(np.array(2.0 ** (i / 32), np.float64).view(np.uint64)) - ((i << 52) // 32)
        assert int(ex[i]) == want, i
    for i in range(16):
        invc, logc = float(lg[2 * i]), float(lg[2 * i + 1])
        assert abs(logc + math.log2(invc)) < 2.0 ** -45, i
        # subinterval i of the reduced argument z in [OFF, 2 OFF), OFF = 0x3f330000 as float bits (about 0.7)
        lo = float(np.array(0x3f330000 + (i << 19), np.uint32).view(F32))
        hi = float(np.array(0x3f330000 + ((i + 1) << 19), np.uint32).view(F32))
        assert lo <= 1 / invc <= hi, i


@pytest.mark.parametrize("ns", GOLDEN_NS)
def test_every_x_in_0_to_1_for_the_reference_exponents(shim, ns):
    """every float x in [0, 1.0001], subnormals included, for every Ns of the reference's scenes"""
    assert {1.0, 10.0, 200.0, 1000.0, 1024.0} <= set(GOLDEN_NS)
    n, rep = check_range(shim, 0, ONE_PLUS, 1, ns)
    assert n == 0, _report(n, rep, f"y = {ns}")


@pytest.mark.parametrize("y", EDGE_Y, ids=repr)
def test_every_5th_float_for_edge_exponents(shim, y):
    """every 5th float bit pattern (negative, subnormal, inf and NaN x included) plus every float in [0.99, 1.0001]"""
    n, rep = check_range(shim, 0, 0xFFFFFFFF, 5, y)
    assert n == 0, _report(n, rep, f"y = {y}, every 5th float")
    n, rep = check_range(shim, fbits(0.99), ONE_PLUS, 1, y)
    assert n == 0, _report(n, rep, f"y = {y}, x in [0.99, 1.0001]")


def test_random_pairs(shim):
    x, y = random_pairs(10_000_000, 7)
    rep = np.zeros(4 * MAX_REP, F32)
    n = shim.strict_host_powf_check_pairs(len(x), x.ctypes.data_as(F32P), y.ctypes.data_as(F32P), PORT, N_THREADS,
                                          rep.ctypes.data_as(F32P), MAX_REP)
    assert n == 0, _report(n, rep, "random pairs")
    # the pairs do reach the special branches
    with np.errstate(all="ignore"):
        r = np.power(x.astype(np.float64), y.astype(np.float64))
        assert (np.isnan(r) & ~np.isnan(x) & ~np.isnan(y)).sum() > 100_000  # negative x, non-integer y
        assert (np.isinf(r) & np.isfinite(x)).sum() > 100_000 and ((r == 0) & (x != 0)).sum() > 100_000
        assert ((x < 0) & (y == np.round(y)) & np.isfinite(r) & (r != 0)).sum() > 100_000


def test_the_old_formula_fails_the_same_harness(shim):
    """(float)pow((double)x, (double)y), what the shading computed before, is not libm's powf"""
    n, _ = check_range(shim, 0, ONE_PLUS, 1, 10.0, OLD_FORMULA)
    assert n > 1000, n
    n, _ = check_range(shim, fbits(0.5), ONE_PLUS, 1, 2.0, OLD_FORMULA)
    assert n > 0, n


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def restated_old_powf(tmp_path_factory, restated):
    """oracle/restated.c built with its one powf call replaced by the old formula"""
    import oracle

    d = tmp_path_factory.mktemp("restated_old_powf")
    src = open(os.path.join(ROOT, "oracle", "restated.c")).read()
    call = "powf(dot3(N, Hh), Ns)"
    assert src.count(call) == 1 and src.count("powf(") == 1
    (d / "restated.c").write_text(src.replace(call, "(float)pow((double)dot3(N, Hh), (double)Ns)"))
    shutil.copy(os.path.join(ROOT, "oracle", "restated.h"), d / "restated.h")
    so = d / "librestated_old_powf.so"
    r = subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-o", str(so),
                        str(d / "restated.c"), "-lm"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    saved = oracle.RESTATED_SO
    oracle.RESTATED_SO = str(so)
    try:
        return oracle.Restated()
    finally:
        oracle.RESTATED_SO = saved


@pytest.mark.parametrize("name", ["c3_water_1080p", "c3_sphere_1080p"])
def test_reference_frames_see_the_old_formula(shim, restated_old_powf, name):
    """rendered with the old formula, the reference's C3 frames miss their float accumulator digest
    (test_fullsize_cpu.py shows that the restatement with libm powf matches it)"""
    from test_fullsize_cpu import _load_full

    sc, z = _load_full(name)
    W, H = int(z["W"]), int(z["H"])
    if not restated_old_powf.set_simd(True):
        pytest.skip("no AVX2 on this host: the scalar restatement needs minutes at this size")
    try:
        o = restated_old_powf.render(to_flat(sc), z["cam"], W, H, faceid=z["faceid"].astype(np.int32))
    finally:
        restated_old_powf.set_simd(False)
    assert np.array_equal(o.tri, z["tri"]) and _sha(o.t) == str(z["sha_t"])
    assert _sha(o.rgb) != str(z["sha_rgb"])


def test_specular_scene_sees_the_old_formula(shim, restated, restated_old_powf):
    """the specular scene of tests/test_gpu_specular.py: the old formula changes its float accumulator"""
    from specular_scene import EYE, LOOK, SEED, specular_scene

    from esctp1raytracer_b200 import Camera, hash_faceids

    s = specular_scene()
    W, H = 320, 240
    cam = Camera.for_frame(EYE, LOOK, W, H)
    fid = hash_faceids(SEED, W, H, s.faces_per_light)
    a = restated.render(to_flat(s), cam.as_array(), W, H, faceid=fid)
    b = restated_old_powf.render(to_flat(s), cam.as_array(), W, H, faceid=fid)
    assert np.array_equal(a.tri, b.tri) and np.array_equal(a.occ_tri, b.occ_tri)
    differ = (a.rgb.view(np.uint32) != b.rgb.view(np.uint32)).any(axis=1).sum()
    assert differ >= 10, differ
