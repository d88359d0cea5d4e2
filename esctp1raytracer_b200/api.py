"""Host-side mirror of the reference's interface for the render path.

Reference                                   here
------------------------------------------  -----------------------------------
tracer::scene (src/scene/scene.h:9-44)      Scene  (flat SoA, reference order)
tracer::camera(lookfrom, lookat, vup,       Camera(lookfrom, lookat, vup, vfov,
  vfov, aspect)  (src/scene/camera.h:16)      aspect)
ispc::trace(W, H, cam, tris, lights, ...,   Renderer.trace(scene, cam, W, H) ->
  image)  (src/ispc/trace.ispc:86-92,         packed u8 RGB rows in PPM order
  called at src/main.cpp:619-624)
scan_row + PPM quantiser                    (what trace() computes)
  (src/main.cpp:698-791, 679-684)

Everything computes on the GPU through the C ABI in include/tracer_cuda.h;
there is no CPU path here.
"""
from __future__ import annotations

import ctypes as C
import operator
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import TracerError

RNG_HASH, RNG_MT19937, RNG_EXPLICIT = 0, 1, 2


def _ptr(a, ctype):
    return None if a is None else a.ctypes.data_as(C.POINTER(ctype))


@dataclass
class Scene:
    """Flat scene in the reference's iteration order: geometry major, face minor
    (src/main.cpp:179-180).  ``geom_material`` rows are ka[3] kd[3] ks[3] ke[3] Ns
    (src/scene/scene.h:11-18); ``light_geom`` is ``light_sources`` (scene.h:38)."""

    geom_tri_offset: np.ndarray
    tri_verts: np.ndarray
    geom_material: np.ndarray
    light_geom: np.ndarray
    tri_normals: np.ndarray | None = None
    geom_has_normals: np.ndarray | None = None
    sphere_cr: np.ndarray = field(default_factory=lambda: np.zeros((0, 4), np.float32))
    sphere_material: np.ndarray = field(default_factory=lambda: np.zeros((0, 13), np.float32))

    def __post_init__(self):
        self.geom_tri_offset = np.ascontiguousarray(self.geom_tri_offset, np.int32)
        self.tri_verts = np.ascontiguousarray(self.tri_verts, np.float32).reshape(-1, 3, 3)
        self.geom_material = np.ascontiguousarray(self.geom_material, np.float32).reshape(-1, 13)
        self.light_geom = np.ascontiguousarray(self.light_geom, np.int32).reshape(-1)
        if self.tri_normals is not None:
            self.tri_normals = np.ascontiguousarray(self.tri_normals, np.float32).reshape(-1, 3, 3)
        if self.geom_has_normals is None:
            self.geom_has_normals = np.zeros(self.n_geoms, np.int32)
        self.geom_has_normals = np.ascontiguousarray(self.geom_has_normals, np.int32)
        self.sphere_cr = np.ascontiguousarray(self.sphere_cr, np.float32).reshape(-1, 4)
        self.sphere_material = np.ascontiguousarray(self.sphere_material, np.float32).reshape(-1, 13)
        if len(self.geom_tri_offset) < 1 or self.geom_tri_offset[-1] != len(self.tri_verts):
            raise ValueError("geom_tri_offset[-1] must equal the triangle count")
        if len(self.geom_material) != self.n_geoms:
            raise ValueError("one material row per geometry")
        if self.geom_has_normals.any() and (self.tri_normals is None or len(self.tri_normals) != self.n_tris):
            raise ValueError("geom_has_normals set but tri_normals missing")

    @property
    def n_geoms(self):
        return len(self.geom_tri_offset) - 1

    @property
    def n_tris(self):
        return int(self.geom_tri_offset[-1])

    @property
    def n_lights(self):
        return len(self.light_geom)

    @property
    def faces_per_light(self):
        o = self.geom_tri_offset
        return np.array([o[g + 1] - o[g] for g in self.light_geom], np.int64)

    @staticmethod
    def load_obj(path: str) -> "Scene":
        """model::loadobj (src/scene/sceneloader.cpp:14-106): OBJ/MTL -> scene, through the library's own
        C++ loader (csrc/host_io.cpp).  Raises TracerError where the reference throws (e.g. any
        loader warning, sceneloader.cpp:27-30)."""
        lib = _lib.load()
        h = C.c_void_p()
        if lib.tracer_scene_load_obj(path.encode(), C.byref(h)) != 0:
            raise TracerError(lib.tracer_host_last_error().decode())
        try:
            return Scene._from_host(lib, h)
        finally:
            lib.tracer_scene_host_free(h)

    @staticmethod
    def _from_host(lib, h) -> "Scene":
        f = lib.tracer_scene_host_flat(h).contents
        G = f.n_geoms
        off = np.ctypeslib.as_array(f.geom_tri_offset, (G + 1,)).copy()
        N = int(off[-1])
        grab = lambda ptr, shape, dt: (np.ctypeslib.as_array(ptr, shape).astype(dt).copy() if int(np.prod(shape)) and ptr else np.zeros(shape, dt))
        hasn = grab(f.geom_has_normals, (G,), np.int32)
        return Scene(off, grab(f.tri_verts, (N, 3, 3), np.float32), grab(f.geom_material, (G, 13), np.float32),
                     grab(f.light_geom, (f.n_lights,), np.int32),
                     tri_normals=grab(f.tri_normals, (N, 3, 3), np.float32) if hasn.any() else None, geom_has_normals=hasn)

    def flatten_sorted(self):
        """flatten_scene (src/simplify/flatten.cpp:50-82): flat triangle array sorted by vertices[0].x, through the
        library's host helper (tracer_scene_flatten_sorted).  Returns (Scene in sorted iteration order,
        origin_geom [N'], origin_prim [N']) — the (geom_id, prim_id) every sorted triangle keeps (flatten.cpp:62-63)."""
        lib = _lib.load()
        h = C.c_void_p()
        cs = self.c_struct()
        if lib.tracer_scene_flatten_sorted(C.byref(cs), C.byref(h)) != 0:
            raise TracerError(lib.tracer_host_last_error().decode())
        try:
            sc = Scene._from_host(lib, h)
            pg, pp = C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)()
            _lib.check(lib.tracer_scene_host_origin(h, C.byref(pg), C.byref(pp)))
            return sc, np.ctypeslib.as_array(pg, (sc.n_tris,)).copy(), np.ctypeslib.as_array(pp, (sc.n_tris,)).copy()
        finally:
            lib.tracer_scene_host_free(h)

    def c_struct(self) -> _lib.SceneFlat:
        s = _lib.SceneFlat()
        s.n_geoms = self.n_geoms
        s.geom_tri_offset = _ptr(self.geom_tri_offset, C.c_int32)
        s.tri_verts = _ptr(self.tri_verts, C.c_float)
        s.tri_normals = _ptr(self.tri_normals, C.c_float)
        s.geom_has_normals = _ptr(self.geom_has_normals, C.c_int32)
        s.geom_material = _ptr(self.geom_material, C.c_float)
        s.n_lights = self.n_lights
        s.light_geom = _ptr(self.light_geom, C.c_int32)
        s.n_spheres = len(self.sphere_cr)
        s.sphere_cr = _ptr(self.sphere_cr, C.c_float)
        s.sphere_material = _ptr(self.sphere_material, C.c_float)
        return s


class Camera:
    """tracer::camera (src/scene/camera.h:16-29): same constructor arguments, same
    arithmetic (computed by the C library's host helper)."""

    def __init__(self, lookfrom, lookat, vup=(0.0, 1.0, 0.0), vfov=60.0, aspect=4.0 / 3.0):
        lib = _lib.load()
        self.c = _lib.CameraC()
        e = (C.c_float * 3)(*[float(x) for x in lookfrom])
        l = (C.c_float * 3)(*[float(x) for x in lookat])
        u = (C.c_float * 3)(*[float(x) for x in vup])
        lib.tracer_camera_lookat(e, l, u, C.c_float(vfov), C.c_float(float(np.float32(aspect))), C.byref(self.c))

    @staticmethod
    def for_frame(lookfrom, lookat, width, height):
        """The camera main() builds: vfov 60, vup (0,1,0), aspect = float(W)/H (main.cpp:548-551)."""
        return Camera(lookfrom, lookat, (0, 1, 0), 60.0, np.float32(width) / np.float32(height))

    def as_array(self):
        return np.array(list(self.c.origin) + list(self.c.lower_left_corner) + list(self.c.horizontal)
                        + list(self.c.vertical), np.float32)


def hash_faceids(seed: int, width: int, height: int, faces_per_light) -> np.ndarray:
    """numpy mirror of the device's counter-based faceID (kernels.cuh:hash_faceid):
    [H*W, L] in image index order h*W+w."""

    def mix(x):
        x = x.astype(np.uint32)
        x ^= x >> np.uint32(16)
        x = (x * np.uint32(0x7FEB352D)).astype(np.uint32)
        x ^= x >> np.uint32(15)
        x = (x * np.uint32(0x846CA68B)).astype(np.uint32)
        x ^= x >> np.uint32(16)
        return x

    with np.errstate(over="ignore"):
        idx = np.arange(width * height, dtype=np.uint32)
        base = mix(np.uint32((seed ^ 0x9E3779B9) & 0xFFFFFFFF) + idx)
        out = np.zeros((width * height, len(faces_per_light)), np.int32)
        for l, F in enumerate(faces_per_light):
            k = np.uint32((l * 0x85EBCA6B + 0xC2B2AE35) & 0xFFFFFFFF)
            h = mix(base ^ k)
            out[:, l] = ((h.astype(np.uint64) * np.uint64(F)) >> np.uint64(32)).astype(np.int32)
    return out


def band_row_count(height, band_rows, band_index, band_count) -> int:
    return int(_lib.load().tracer_band_row_count(height, band_rows, band_index, band_count))


def _crop_window(crop, width, height, bands):
    """(x, y, w, h) of a crop window inside the width x height frame, or ValueError"""
    try:
        x, y, w, h = (operator.index(c) for c in crop)
    except (TypeError, ValueError):
        raise ValueError(f"crop must be four integers (x, y, w, h), not {crop!r}") from None
    if w < 1 or h < 1 or x < 0 or y < 0 or x + w > width or y + h > height:
        raise ValueError(f"crop window {(x, y, w, h)} is not inside the {width} x {height} frame")
    if bands is not None:
        raise ValueError("a crop window does not combine with bands")
    return x, y, w, h


@dataclass
class Frame:
    rgb8: np.ndarray  # [rows, W, 3] uint8, PPM row order (row 0 = h=H-1)
    stats: dict
    tri: np.ndarray | None = None
    t: np.ndarray | None = None
    v: np.ndarray | None = None
    occ_tri: np.ndarray | None = None
    rgb: np.ndarray | None = None


_UPDATE_ROW = dict(tri_verts=9, tri_normals=9, geom_material=13, sphere_cr=4, sphere_material=13)


def _update_rows(name, shape, row):
    """rows of an update array: shape [n, row] (triangles also [n, 3, 3]) or flat [n * row]"""
    size = int(np.prod(shape)) if len(shape) else -1
    if size < 0 or size % row or (len(shape) > 1 and int(np.prod(shape[1:])) != row):
        raise ValueError(f"{name}: shape {tuple(shape)} is not [n, {row}]")
    return size // row


def _update_array(name, a):
    """(address, rows, on the device, interface stream or None, object to keep alive) of one update argument.  A host array
    is converted like Scene's arrays (C-contiguous float32); an object with __cuda_array_interface__ is read in place, so
    it must already be float32 and C-contiguous."""
    row = _UPDATE_ROW[name]
    cai = getattr(a, "__cuda_array_interface__", None)
    if cai is None:
        h = np.ascontiguousarray(a, np.float32)
        return h.ctypes.data, _update_rows(name, h.shape, row), False, None, h
    shape = tuple(int(x) for x in cai["shape"])
    if np.dtype(cai["typestr"]) != np.dtype(np.float32):
        raise ValueError(f"{name}: device arrays must be float32, not {cai['typestr']}")
    strides = cai.get("strides")
    if strides is not None:
        want = [4 * int(np.prod(shape[i + 1:])) for i in range(len(shape))]
        if any(n > 1 and int(s) != w for n, s, w in zip(shape, strides, want)):
            raise ValueError(f"{name}: device arrays must be C-contiguous (strides {tuple(strides)})")
    return int(cai["data"][0]), _update_rows(name, shape, row), True, cai.get("stream"), a


def _scene_update(scene: Scene, *, tri_verts=None, first_tri=0, tri_normals=None, geom_material=None, sphere_cr=None,
                  sphere_material=None, stream=None):
    """The tracer_scene_update of an update() call and the objects it points into.  Needs no device: every check that can
    be made from shapes and types is made here; the library checks the range and, for device arrays, the pointers."""
    u = _lib.SceneUpdate()
    u.struct_size = C.sizeof(_lib.SceneUpdate)
    given = dict(tri_verts=tri_verts, tri_normals=tri_normals, geom_material=geom_material, sphere_cr=sphere_cr,
                 sphere_material=sphere_material)
    keep, rows, on_device, streams = [], {}, set(), set()
    for name, a in given.items():
        if a is None:
            continue
        ptr, rows[name], dev, st, k = _update_array(name, a)
        keep.append(k)
        on_device.add(dev)
        if st is not None:
            streams.add(int(st))
        setattr(u, name, ptr or None)
    if len(on_device) > 1:
        raise ValueError("an update takes host arrays or device arrays, not both")
    n_tri = {rows[k] for k in ("tri_verts", "tri_normals") if k in rows}
    if len(n_tri) > 1:
        raise ValueError("tri_verts and tri_normals cover different numbers of triangles")
    n_sph = len(scene.sphere_cr)
    for name, want in (("geom_material", scene.n_geoms), ("sphere_cr", n_sph), ("sphere_material", n_sph)):
        if name in rows and rows[name] != want:
            raise ValueError(f"{name}: {rows[name]} rows, the scene has {want}")
    if not -2 ** 31 <= int(first_tri) < 2 ** 31:
        raise ValueError("first_tri out of range")
    u.tri_first, u.tri_count = int(first_tri), (n_tri.pop() if n_tri else 0)
    u.data_is_device = int(on_device == {True})
    if stream is not None:
        u.cuda_stream = int(stream)
    elif u.data_is_device:
        if len(streams) > 1:
            raise ValueError("device arrays name different streams: pass stream=")
        # no stream in the interface (torch's has none): the legacy default stream, behind work queued on it
        u.cuda_stream = streams.pop() if streams else 1
    return u, keep


_UPDATE_DOC = """Replace vertices, normals, materials or spheres in place (tracer_cuda_scene_update{multi}); topology stays.

        ``tri_verts`` / ``tri_normals``: [n, 3, 3] for triangles ``[first_tri, first_tri + n)`` (normals only for a scene
        created with them); ``geom_material`` [n_geoms, 13]; ``sphere_cr`` [n_spheres, 4]; ``sphere_material``
        [n_spheres, 13].  Each is a host array (converted to float32) or an object with ``__cuda_array_interface__`` such
        as a torch CUDA tensor on {device} (float32, C-contiguous, read in place); one call takes one kind.  The copies
        run on ``stream`` (a cudaStream_t handle), else on the interface's ``stream`` entry, else, for device arrays, on
        the legacy default stream, so data written there first is ordered before them; a tensor written on another
        stream needs that stream here.  The call returns when the update is complete on the device.  The next frame is
        the frame a fresh upload of the updated arrays gives, bit for bit.

        ``self.scene`` keeps describing the topology, which is all ``trace`` reads from it: its arrays are those of the
        upload and are not kept in sync with updates.  Raises ValueError for a wrong shape or dtype, a non-contiguous
        device array or host and device arrays mixed; TracerError when the library refuses the update (range outside
        the scene, normals for a scene without them, a pointer not on {device}), which leaves the scene unchanged."""


class ResidentScene:
    """A scene uploaded to HBM (tracer_cuda_scene_create)."""

    def __init__(self, renderer, scene: Scene):
        self.renderer = renderer
        self.scene = scene
        self.handle = C.c_void_p()
        cs = scene.c_struct()
        _lib.check(renderer.lib.tracer_cuda_scene_create(C.byref(cs), C.byref(self.handle)))

    def update(self, *, tri_verts=None, first_tri=0, tri_normals=None, geom_material=None, sphere_cr=None,
               sphere_material=None, stream=None):
        # keep: the arrays u points into, alive for the call
        u, keep = _scene_update(self.scene, tri_verts=tri_verts, first_tri=first_tri, tri_normals=tri_normals,
                                geom_material=geom_material, sphere_cr=sphere_cr, sphere_material=sphere_material,
                                stream=stream)  # noqa: F841
        _lib.check(self.renderer.lib.tracer_cuda_scene_update(self.handle, C.byref(u)))

    update.__doc__ = _UPDATE_DOC.format(multi="", device="the scene's GPU")

    def close(self):
        if self.handle:
            self.renderer.lib.tracer_cuda_scene_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiRenderer:
    """All GPUs of the box behind one call, one process (tracer_cuda_init_multi): interleaved 8-row bands, scene
    replicated, packed bands gathered on GPU 0 with NCCL inside the library.  The multi-process form (one rank per
    GPU, torch.distributed) lives in dist.py; both produce the bytes a single GPU produces."""

    def __init__(self, n_gpus: int):
        self.lib = _lib.load()
        _lib.check(self.lib.tracer_cuda_init_multi(n_gpus))
        self.n_gpus = n_gpus

    def upload(self, scene: Scene):
        h = C.c_void_p()
        cs = scene.c_struct()
        _lib.check(self.lib.tracer_cuda_scene_create_multi(C.byref(cs), C.byref(h)))
        return _MultiScene(self, scene, h)

    def trace(self, scene, camera: "Camera", width: int, height: int, *, rng_mode=RNG_HASH, seed=1, faceid=None,
              samples_per_pixel=0, bundle_cull=False, band_rows=0, out_device_ptr=None, bvh=False) -> "Frame":
        """``out_device_ptr``: leave the assembled frame in HBM on GPU 0 at that address instead of copying it to the host.
        ``bvh``: the optional BVH mode (opts.accel = 1; every GPU builds its replica's tree), same bytes."""
        sc = scene.scene if isinstance(scene, _MultiScene) else scene
        o = _lib.RenderOpts()
        o.struct_size = C.sizeof(_lib.RenderOpts)
        o.rng_mode, o.seed = rng_mode, seed & 0xFFFFFFFF
        keep = None
        if rng_mode == RNG_EXPLICIT:
            keep = np.ascontiguousarray(faceid, np.int32)
            o.faceid = _ptr(keep, C.c_int32)
        o.samples_per_pixel, o.bundle_cull, o.band_rows = samples_per_pixel, int(bundle_cull), band_rows
        o.accel = int(bool(bvh))
        if out_device_ptr is not None:
            out, dst, o.rgb_out_is_device = None, C.c_void_p(out_device_ptr), 1
        else:
            out = np.empty((height, width, 3), np.uint8)
            dst = out.ctypes.data_as(C.c_void_p)
        stats = {}
        if isinstance(scene, _MultiScene):
            _lib.check(self.lib.tracer_cuda_render_scene_multi(scene.handle, C.byref(camera.c), width, height, C.byref(o), dst))
            st = _lib.FrameStats()
            _lib.check(self.lib.tracer_cuda_last_stats_multi(scene.handle, C.byref(st)))
            stats = st.asdict()
        else:
            cs = sc.c_struct()
            _lib.check(self.lib.tracer_cuda_render_multi(C.byref(cs), C.byref(camera.c), width, height, C.byref(o), dst))
        return Frame(rgb8=out, stats=stats)


class _MultiScene:
    def __init__(self, renderer, scene, handle):
        self.renderer, self.scene, self.handle = renderer, scene, handle

    def update(self, *, tri_verts=None, first_tri=0, tri_normals=None, geom_material=None, sphere_cr=None,
               sphere_material=None, stream=None):
        # keep: the arrays u points into, alive for the call
        u, keep = _scene_update(self.scene, tri_verts=tri_verts, first_tri=first_tri, tri_normals=tri_normals,
                                geom_material=geom_material, sphere_cr=sphere_cr, sphere_material=sphere_material,
                                stream=stream)  # noqa: F841
        _lib.check(self.renderer.lib.tracer_cuda_scene_update_multi(self.handle, C.byref(u)))

    update.__doc__ = _UPDATE_DOC.format(multi="_multi", device="GPU 0") + """  Every replica is updated; a refused
        update changes none."""

    def close(self):
        if self.handle:
            self.renderer.lib.tracer_cuda_scene_destroy_multi(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Renderer:
    """One CUDA device (tracer_cuda_init); see MultiRenderer for all GPUs of the box in one process."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        _lib.check(self.lib.tracer_cuda_init(device))
        self.device = device

    def device_info(self) -> dict:
        d = _lib.DeviceInfo()
        _lib.check(self.lib.tracer_cuda_device_info(C.byref(d)))
        return dict(name=d.name.decode(), sm_count=d.sm_count, cc=(d.cc_major, d.cc_minor), clock_khz=d.clock_khz,
                    total_mem=d.total_mem, l2_bytes=d.l2_bytes)

    def upload(self, scene: Scene) -> ResidentScene:
        return ResidentScene(self, scene)

    def _opts(self, scene, width, height, rng_mode, seed, faceid, bands, exhaustive, debug, n_px, keep, tuning, n_views=1):
        o = _lib.RenderOpts()
        o.struct_size = C.sizeof(_lib.RenderOpts)
        o.rng_mode, o.seed = rng_mode, seed & 0xFFFFFFFF
        if rng_mode == RNG_EXPLICIT:
            f = np.ascontiguousarray(faceid, np.int32)
            if f.size != n_views * width * height * scene.n_lights:
                raise ValueError("faceid must have W*H*n_lights entries (image index order)")
            keep.append(f)
            o.faceid = _ptr(f, C.c_int32)
        if bands is not None:
            o.band_rows, o.band_index, o.band_count = bands
        o.exhaustive_strict = int(exhaustive)
        o.rays_per_thread, o.shadow_chunks, o.samples_per_pixel, o.bundle_cull, o.accel = tuning
        dbg = {}
        if debug:
            L = scene.n_lights
            dbg = dict(tri=np.zeros(n_px, np.int32), t=np.zeros(n_px, np.float32), v=np.zeros(n_px, np.float32),
                       occ_tri=np.full((n_px, L), -2, np.int32), rgb=np.zeros((n_px, 3), np.float32))
            o.out_tri, o.out_t, o.out_v = _ptr(dbg["tri"], C.c_int32), _ptr(dbg["t"], C.c_float), _ptr(dbg["v"], C.c_float)
            o.out_occ_tri, o.out_rgb = _ptr(dbg["occ_tri"], C.c_int32), _ptr(dbg["rgb"], C.c_float)
        return o, dbg

    def trace(self, scene, camera: Camera, width: int, height: int, *, rng_mode=RNG_HASH, seed=1, faceid=None,
              bands=None, exhaustive_strict=False, debug=False, out_device_ptr=None, stream=None,
              rays_per_thread=0, shadow_chunks=0, samples_per_pixel=0, bundle_cull=False, out=None, bvh=False,
              row_hits_exchange=None, crop=None) -> Frame:
        """Render; ``scene`` is a Scene (one-shot: upload + render, the drop-in call) or a
        ResidentScene.  ``bvh``: the optional BVH mode (opts.accel = 1): the resident scene builds its tree on the
        first such render and keeps it; same bytes as the default mode.  ``bands`` = (band_rows, band_index, band_count).  With
        ``out_device_ptr`` the packed rows are left in HBM at that address; ``out`` is an optional
        caller-owned uint8 [rows, W, 3] host array (e.g. pinned) to receive them.  ``row_hits_exchange``: with
        ``RNG_MT19937`` and bands, a callable ``(row_hits: np.ndarray[int32, H]) -> None`` that completes this call's
        per-row hit counts into the frame's, in place (opts.row_hits_exchange; an all-reduce sum over the calls that render
        the frame does it).  An exception inside it fails the render with TracerError.

        ``crop`` = (x, y, w, h): render only columns [x, x+w) of PPM rows [y, y+h) (row 0 at the top) of the width x
        height frame.  ``rgb8`` is then [h, w, 3] and the debug arrays [h*w, ...], bit for bit the same pixels of the whole
        frame, in every mode; ``faceid`` (RNG_EXPLICIT) stays the whole frame's.  Raises ValueError for a window that is not
        inside the frame, a crop with ``bands`` or an ``out`` that is not uint8 [h, w, 3], before any library call."""
        window = None if crop is None else _crop_window(crop, width, height, bands)
        if window is not None and out is not None and out_device_ptr is None and (
                out.dtype != np.uint8 or out.shape != (window[3], window[2], 3) or not out.flags.c_contiguous):
            raise ValueError(f"out must be a C-contiguous uint8 array of shape ({window[3]}, {window[2]}, 3)")
        sc = scene.scene if isinstance(scene, ResidentScene) else scene
        rows = height if bands is None else band_row_count(height, *bands)
        cols = width
        if window is not None:
            cols, rows = window[2], window[3]
        n_px = rows * cols
        keep = []
        o, dbg = self._opts(sc, width, height, rng_mode, seed, faceid, bands, exhaustive_strict, debug, n_px, keep,
                            (rays_per_thread, shadow_chunks, samples_per_pixel, int(bundle_cull), int(bool(bvh))))
        if window is not None:
            o.crop_x, o.crop_y, o.crop_w, o.crop_h = window
        if out_device_ptr is not None:
            out = None
            o.rgb_out_is_device = 1
            dst = C.c_void_p(out_device_ptr)
        else:
            if out is None:
                out = np.zeros((rows, cols, 3), np.uint8)
            assert out.dtype == np.uint8 and out.size == rows * cols * 3 and out.flags.c_contiguous
            dst = out.ctypes.data_as(C.c_void_p)
        if stream is not None:
            o.cuda_stream = C.c_void_p(stream)
        if row_hits_exchange is not None:
            o.row_hits_exchange = keep_cb = _row_hits_hook(row_hits_exchange)  # noqa: F841 (alive for the call)
        stats = {}
        if isinstance(scene, ResidentScene):
            _lib.check(self.lib.tracer_cuda_render_scene(scene.handle, C.byref(camera.c), width, height, C.byref(o), dst))
            st = _lib.FrameStats()
            _lib.check(self.lib.tracer_cuda_last_stats(scene.handle, C.byref(st)))
            stats = st.asdict()
        else:
            cs = sc.c_struct()
            _lib.check(self.lib.tracer_cuda_render(C.byref(cs), C.byref(camera.c), width, height, C.byref(o), dst))
        return Frame(rgb8=out, stats=stats, **dbg)

    def trace_views(self, scene: ResidentScene, cameras, width: int, height: int, *, rng_mode=RNG_HASH, seed=1,
                    faceid=None, exhaustive_strict=False, debug=False, out_device_ptr=None, stream=None, rays_per_thread=0,
                    shadow_chunks=0, samples_per_pixel=0, out=None, bvh=False) -> Frame:
        """Render one view per camera of a ResidentScene in one call (tracer_cuda_render_views).  View v is bit for bit
        ``trace(scene, cameras[v], width, height, ...)`` with the same options; the views share the frame's
        camera-independent work (shadow sweeps, sorts, quantise, read-backs).  ``cameras``: a non-empty sequence of
        Camera.  ``rgb8`` is [V, H, W, 3] (PPM row order per view); with ``debug`` the arrays are [V, H*W, ...].
        ``faceid`` (RNG_EXPLICIT): [V, W*H*L] or [V, H*W, L], image index order per view.  ``out``: optional uint8
        [V, H, W, 3] host array; ``out_device_ptr``: leave the V packed frames in HBM at that address.  Raises
        ValueError for a wrong shape before any library call."""
        if not isinstance(scene, ResidentScene):
            raise ValueError("trace_views renders a ResidentScene (Renderer.upload)")
        cams = list(cameras) if not isinstance(cameras, Camera) else None
        if not cams or not all(isinstance(c, Camera) for c in cams):
            raise ValueError("cameras must be a non-empty sequence of Camera")
        V, sc, L = len(cams), scene.scene, scene.scene.n_lights
        if width < 2 or height < 2:
            raise ValueError("width and height must be >= 2")
        n_px = width * height
        if rng_mode == RNG_EXPLICIT:
            shape = np.shape(faceid)
            if shape not in ((V, n_px * L), (V, n_px, L)):
                raise ValueError(f"faceid must be [V, W*H*L] or [V, H*W, L] = [{V}, {n_px * L}] or [{V}, {n_px}, {L}], "
                                 f"not {list(shape)}")
        keep = []
        o, dbg = self._opts(sc, width, height, rng_mode, seed, faceid, None, exhaustive_strict, debug, V * n_px, keep,
                            (rays_per_thread, shadow_chunks, samples_per_pixel, 0, int(bool(bvh))), n_views=V)
        if out_device_ptr is not None:
            out = None
            o.rgb_out_is_device = 1
            dst = C.c_void_p(out_device_ptr)
        else:
            if out is None:
                out = np.zeros((V, height, width, 3), np.uint8)
            if out.dtype != np.uint8 or out.shape != (V, height, width, 3) or not out.flags.c_contiguous:
                raise ValueError(f"out must be a C-contiguous uint8 array of shape ({V}, {height}, {width}, 3)")
            dst = out.ctypes.data_as(C.c_void_p)
        if stream is not None:
            o.cuda_stream = C.c_void_p(stream)
        carr = (_lib.CameraC * V)(*[c.c for c in cams])
        _lib.check(self.lib.tracer_cuda_render_views(scene.handle, carr, V, width, height, C.byref(o), dst))
        st = _lib.FrameStats()
        _lib.check(self.lib.tracer_cuda_last_stats(scene.handle, C.byref(st)))
        dbg = {k: a.reshape((V, n_px) + a.shape[1:]) for k, a in dbg.items()}
        return Frame(rgb8=out, stats=st.asdict(), **dbg)

    def assemble_bands(self, gathered_ptr, frame_ptr, width, height, band_rows, band_count, rows_pad, stream=None):
        _lib.check(self.lib.tracer_cuda_assemble_bands(C.c_void_p(gathered_ptr), C.c_void_p(frame_ptr), width, height,
                                                       band_rows, band_count, rows_pad,
                                                       C.c_void_p(stream) if stream else None))

    def fp32_peak(self, variant=0, iters=10):
        tf, ms = C.c_double(), C.c_double()
        _lib.check(self.lib.tracer_cuda_fp32_peak(variant, iters, C.byref(tf), C.byref(ms)))
        return tf.value, ms.value


def _row_hits_hook(fn):
    """opts.row_hits_exchange over a Python callable.  ctypes would print an exception raised in a callback and return 0,
    which the library would read as success: it returns 1 instead."""

    def hook(_user, height, rows):
        try:
            fn(np.ctypeslib.as_array(rows, (height,)))
            return 0
        except BaseException:  # noqa: BLE001 — any failure must reach the library as a non-zero return
            import traceback

            traceback.print_exc()
            return 1

    return _lib.ROW_HITS_EXCHANGE(hook)


def write_ppm(path: str, rgb8: np.ndarray, binary: bool = False) -> None:
    """The reference's PPM writer (src/main.cpp:658-689): ASCII P3, rows top to bottom; P6 when binary."""
    a = np.ascontiguousarray(rgb8, np.uint8)
    h, w = a.shape[0], a.shape[1]
    lib = _lib.load()
    if lib.tracer_write_ppm(path.encode(), a.ctypes.data_as(C.c_void_p), w, h, int(binary)) != 0:
        raise TracerError(lib.tracer_host_last_error().decode())


def mt19937_faceids(scene: Scene, width: int, height: int, seed: int, hit_mask) -> np.ndarray:
    """std::mt19937 replay of scan_row's draws (host; tracer_mt19937_faceids)."""
    lib = _lib.load()
    hit = np.ascontiguousarray(hit_mask, np.uint8).reshape(-1)
    out = np.full((width * height, scene.n_lights), -1, np.int32)
    cs = scene.c_struct()
    _lib.check(lib.tracer_mt19937_faceids(C.byref(cs), width, height, seed & 0xFFFFFFFF, _ptr(hit, C.c_uint8),
                                          _ptr(out, C.c_int32)))
    return out
