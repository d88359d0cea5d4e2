"""Crop windows without a device: the RenderOpts layout of the crop fields against the C header, and the argument checks
that Renderer.trace and the CLI make before any library call."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT

from esctp1raytracer_b200 import Camera, Renderer, _lib, scenes

W, H = 120, 80


def test_crop_fields_match_c_layout(tmp_path):
    src = tmp_path / "crop.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "tracer_cuda.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(tracer_render_opts), offsetof(tracer_render_opts, row_hits_user),'
        'offsetof(tracer_render_opts, crop_x), offsetof(tracer_render_opts, crop_y), offsetof(tracer_render_opts, crop_w),'
        'offsetof(tracer_render_opts, crop_h));return 0;}\n')
    exe = tmp_path / "crop"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    O = _lib.RenderOpts
    assert got == [C.sizeof(O), O.row_hits_user.offset, O.crop_x.offset, O.crop_y.offset, O.crop_w.offset, O.crop_h.offset]
    assert O.crop_x.offset > O.row_hits_user.offset  # appended: an older struct_size reads as no crop


def _renderer():
    """a Renderer that never initialised a device: trace must refuse before it calls the library"""
    r = Renderer.__new__(Renderer)
    r.lib = None  # any library call would fail with AttributeError, not ValueError
    return r


@pytest.mark.parametrize("crop", [
    (0, 0, 0, 0), (0, 0, 0, 5), (0, 0, 5, 0), (-1, 0, 5, 5), (0, -1, 5, 5), (W - 4, 0, 5, 5), (0, H - 4, 5, 5),
    (0, 0, W + 1, 1), (0, 0, 1, H + 1), (1, 2, 3), (1, 2, 3, 4, 5), (0.5, 0, 4, 4), ("0", 0, 4, 4), 5,
])
def test_trace_refuses_bad_windows(crop):
    s = scenes.box_scene()
    with pytest.raises(ValueError):
        _renderer().trace(s, Camera.for_frame((0, 1, 3), (0, 1, 0), W, H), W, H, crop=crop)


def test_trace_refuses_crop_with_bands_or_wrong_out():
    s = scenes.box_scene()
    cam = Camera.for_frame((0, 1, 3), (0, 1, 0), W, H)
    with pytest.raises(ValueError):
        _renderer().trace(s, cam, W, H, crop=(0, 0, 8, 8), bands=(8, 0, 2))
    for out in (np.zeros((8, 9, 3), np.uint8), np.zeros((9, 8, 3), np.uint8), np.zeros((8, 8, 3), np.float32),
                np.zeros((8, 8 * 3), np.uint8), np.zeros((8, 16, 3), np.uint8)[:, ::2]):
        with pytest.raises(ValueError):
            _renderer().trace(s, cam, W, H, crop=(3, 4, 8, 8), out=out)


def test_other_calls_take_no_crop():
    from esctp1raytracer_b200 import MultiRenderer

    for fn in (Renderer.trace_views, MultiRenderer.trace):
        with pytest.raises(TypeError):
            fn(None, None, None, W, H, crop=(0, 0, 4, 4))


def test_cli_refusals():
    cli = os.path.join(ROOT, "esctp1raytracer_b200", "tracer_cli.bin")
    for extra, word in ((["--eye", "0,1,3"], "--eye"), (["--gpus", "2"], "--gpus"), ([], "width and height")):
        crop = "0,0,0,0" if not extra else "0,0,4,4"
        r = subprocess.run([cli, "-w", f"{W},{H}", "--crop", crop] + extra, capture_output=True, text=True)
        assert r.returncode != 0 and "--crop" in r.stderr and word in r.stderr, r.stderr
    r = subprocess.run([cli, "--crop", "1,2,3"], capture_output=True, text=True)
    assert r.returncode != 0 and "--crop x,y,w,h" in r.stderr
