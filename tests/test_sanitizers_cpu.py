"""SURVEY §5 "race detection / sanitizers", host side: the product's host code (csrc/host_io.cpp — OBJ/MTL loader,
flatten + sort, PPM writer; csrc/tracer_host.cpp — camera, mt19937 replay, band maths) compiled with
AddressSanitizer + UndefinedBehaviorSanitizer and driven by tests/host_san_driver.cpp over the reference's models
(when the reference tree is present) and over hostile OBJ/MTL text.  The reference itself has no sanitizer build
(no -fsanitize anywhere in its CMake files); its loader aborts the process on bad input (uncaught exception,
src/scene/sceneloader.cpp:27-30) where ours returns a status.

(The device side cannot be run under compute-sanitizer on this GPU pool — DESIGN.md §8 — and carries its own
pipeline race check instead, asserted by every GPU test.)
"""
import glob
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "esctp1raytracer_b200", "csrc")
MODELS = "/root/reference/src/models"


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    if not shutil.which("g++"):
        pytest.skip("no g++")
    out = tmp_path_factory.mktemp("san") / "host_san_driver"
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fno-omit-frame-pointer", "-fsanitize=address,undefined",
           "-fno-sanitize-recover=undefined", os.path.join(ROOT, "tests", "host_san_driver.cpp"),
           os.path.join(CSRC, "host_io.cpp"), os.path.join(CSRC, "tracer_host.cpp"), "-o", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0 and "asan" in r.stderr.lower() and "cannot find" in r.stderr.lower():
        pytest.skip("libasan is not installed")
    assert r.returncode == 0, r.stderr
    return str(out)


def run(driver, scratch, models):
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=1:abort_on_error=0:halt_on_error=1", UBSAN_OPTIONS="print_stacktrace=1")
    env.pop("LD_PRELOAD", None)
    r = subprocess.run([driver, str(scratch)] + models, capture_output=True, text=True, env=env, timeout=300)
    report = r.stdout[-2000:] + r.stderr[-6000:]
    assert r.returncode == 0, report
    assert "AddressSanitizer" not in r.stderr and "LeakSanitizer" not in r.stderr and "runtime error" not in r.stderr, report
    assert "no sanitizer report" in r.stdout
    return r.stdout


def test_host_code_clean_under_asan_ubsan_on_hostile_input(driver, tmp_path):
    out = run(driver, tmp_path, [])
    # the plain cases load, the broken ones are refused with a message — none crashes
    loaded, refused = (int(x) for x in out.split("host_san_driver:")[1].replace(",", "").split() if x.isdigit())
    assert loaded >= 10 and refused >= 8


def test_host_code_clean_under_asan_ubsan_on_the_reference_models(driver, tmp_path):
    """the reference's models when its tree is present, and always the stored geometry of the ones in tests/golden (as
    the reference's loader flattened them) written back as OBJ + MTL"""
    from conftest import golden_names, load_golden, write_obj

    def counts(out):  # (scenes loaded, refused)
        return tuple(int(x) for x in out.split("host_san_driver:")[1].replace(",", "").split() if x.isdigit())

    def scratch(name):
        d = tmp_path / name
        d.mkdir()
        return d

    base = counts(run(driver, scratch("base"), []))  # the driver's own cases alone
    golden = []
    for name in golden_names():
        obj = scratch(name) / "scene.obj"
        write_obj(load_golden(name)[0], obj)
        golden.append(str(obj))
    assert counts(run(driver, scratch("golden"), golden)) == (base[0] + len(golden), base[1])  # every one of them loads
    models = sorted(glob.glob(os.path.join(MODELS, "**", "*.obj"), recursive=True))
    if models:
        out = run(driver, scratch("models"), models)
        assert "scenes loaded" in out
