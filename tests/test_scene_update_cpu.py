"""Scene updates (tracer_cuda_scene_update) without a GPU: the tracer_scene_update layout against ctypes, the C entry
point's refusal of a NULL scene, and the Python helper that turns update() arguments into the struct (shapes, dtypes,
contiguity, host/device mixes, the stream), with stand-in device arrays."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT

from esctp1raytracer_b200 import _lib, scenes
from esctp1raytracer_b200.api import _scene_update


class DeviceStandIn:
    """an object that exposes only __cuda_array_interface__, like a CUDA tensor; no memory behind the address"""

    def __init__(self, shape, typestr="<f4", strides=None, ptr=0x7F0000000000, stream=None):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, strides=strides, data=(ptr, False),
                                             version=3)
        if stream is not None:
            self.__cuda_array_interface__["stream"] = stream


@pytest.fixture(scope="module")
def scene():
    return scenes.soup_scene(400, 8, 2, n_spheres=5, seed=3)


def test_struct_layout_matches_c(tmp_path):
    src = tmp_path / "sz.c"
    fields = [f for f, _ in _lib.SceneUpdate._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tracer_cuda.h"\nint main(void){printf("%zu'
                   + " %zu" * len(fields) + '\\n", sizeof(tracer_scene_update)'
                   + "".join(f", offsetof(tracer_scene_update, {f})" for f in fields) + ");return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(_lib.SceneUpdate)] + [getattr(_lib.SceneUpdate, f).offset for f in fields]


def test_null_scene_is_invalid_without_a_device():
    lib = _lib.load()
    u = _lib.SceneUpdate()
    u.struct_size = C.sizeof(u)
    assert lib.tracer_cuda_scene_update(None, C.byref(u)) == -1  # TRACER_ERR_INVALID
    assert b"null" in lib.tracer_cuda_last_error()
    assert lib.tracer_cuda_scene_update_multi(None, C.byref(u)) == -1


def test_host_arrays(scene):
    v = scene.tri_verts[10:20].astype(np.float64)  # converted, as Scene converts
    u, keep = _scene_update(scene, tri_verts=v, first_tri=10, geom_material=scene.geom_material,
                            sphere_cr=scene.sphere_cr.reshape(-1))
    assert u.struct_size == C.sizeof(_lib.SceneUpdate) and u.data_is_device == 0 and not u.cuda_stream
    assert (u.tri_first, u.tri_count) == (10, 10)
    assert u.tri_verts == keep[0].ctypes.data and keep[0].dtype == np.float32 and np.array_equal(keep[0], v.astype(np.float32))
    assert u.geom_material == scene.geom_material.ctypes.data and u.sphere_cr and not u.tri_normals and not u.sphere_material
    u, _ = _scene_update(scene, tri_normals=np.zeros((7, 9), np.float32), first_tri=3)
    assert (u.tri_first, u.tri_count) == (3, 7) and not u.tri_verts
    u, _ = _scene_update(scene)  # nothing: the library's no-op
    assert u.tri_count == 0 and not any(getattr(u, f) for f in ("tri_verts", "tri_normals", "geom_material", "sphere_cr"))
    u, _ = _scene_update(scene, sphere_material=scene.sphere_material, stream=0x1234)
    assert u.cuda_stream == 0x1234


@pytest.mark.parametrize("kw", [
    dict(tri_verts=np.zeros((4, 3, 2), np.float32)),
    dict(tri_verts=np.zeros(10, np.float32)),
    dict(tri_verts=np.zeros((2, 3, 3), np.float32), tri_normals=np.zeros((3, 3, 3), np.float32)),
    dict(geom_material=np.zeros((7, 13), np.float32)),
    dict(geom_material=np.zeros((8, 12), np.float32)),
    dict(sphere_cr=np.zeros((4, 4), np.float32)),
    dict(sphere_material=np.zeros((5, 4), np.float32)),
    dict(tri_verts=np.zeros((1, 9), np.float32), first_tri=2 ** 31),
])
def test_host_shapes_rejected(scene, kw):
    with pytest.raises(ValueError):
        _scene_update(scene, **kw)


def test_device_arrays(scene):
    a = DeviceStandIn((5, 3, 3), ptr=0x1000)
    m = DeviceStandIn((8, 13), ptr=0x2000, strides=(52, 4))  # explicit C strides are fine
    u, _ = _scene_update(scene, tri_verts=a, first_tri=30, geom_material=m)
    assert u.data_is_device == 1 and u.tri_verts == 0x1000 and u.geom_material == 0x2000 and (u.tri_first, u.tri_count) == (30, 5)
    assert u.cuda_stream == 1  # no stream entry (torch's interface has none): the legacy default stream
    u, _ = _scene_update(scene, tri_verts=DeviceStandIn((5, 9), stream=0xABC))
    assert u.cuda_stream == 0xABC
    u, _ = _scene_update(scene, tri_verts=DeviceStandIn((5, 9), stream=0xABC), stream=0xDEF)  # stream= wins
    assert u.cuda_stream == 0xDEF
    u, _ = _scene_update(scene, tri_verts=DeviceStandIn((1, 3, 3), strides=(4, 12, 4)))  # a size-1 dim's stride is free
    assert u.tri_count == 1


@pytest.mark.parametrize("kw", [
    dict(tri_verts=DeviceStandIn((5, 3, 3), typestr="<f8")),
    dict(tri_verts=DeviceStandIn((5, 3, 3), typestr="<i4")),
    dict(tri_verts=DeviceStandIn((5, 3, 3), typestr=">f4")),
    dict(tri_verts=DeviceStandIn((5, 3, 3), strides=(72, 4, 12))),  # transposed
    dict(tri_verts=DeviceStandIn((5, 9), strides=(72, 4))),  # every other row
    dict(tri_verts=DeviceStandIn((5, 8))),
    dict(sphere_cr=DeviceStandIn((5, 3))),
    dict(geom_material=DeviceStandIn((9, 13))),
    dict(tri_verts=DeviceStandIn((5, 9)), geom_material=np.zeros((8, 13), np.float32)),  # host and device mixed
    dict(tri_verts=np.zeros((5, 9), np.float32), sphere_cr=DeviceStandIn((5, 4))),
    dict(tri_verts=DeviceStandIn((5, 9), stream=5), sphere_cr=DeviceStandIn((5, 4), stream=6)),  # two streams
])
def test_device_arrays_rejected(scene, kw):
    with pytest.raises(ValueError):
        _scene_update(scene, **kw)
