"""Resident-scene updates (tracer_cuda_scene_update, ResidentScene.update) on the GPU: after an update every frame equals
the frame of a fresh upload of the updated arrays (packed bytes, hit ids, t, v, first occluders and the float accumulator),
in the default, bundle-cull and BVH modes, with every rng mode and with bands; refused updates change nothing; the box the
device computes equals the host loop it replaced."""
import ctypes as C
import dataclasses
import hashlib

import numpy as np
import pytest

from conftest import bits

pytestmark = pytest.mark.gpu

W, H = 128, 96
EYE, LOOK = (0, 1, 3), (0, 1, 0)
MODES = [dict(), dict(bundle_cull=1), dict(bvh=True)]


@pytest.fixture(scope="module")
def renderer():
    from esctp1raytracer_b200 import Renderer

    return Renderer(0)


def _cam(w=W, h=H):
    from esctp1raytracer_b200 import Camera

    return Camera.for_frame(EYE, LOOK, w, h)


def _same_frames(a, b):
    assert np.array_equal(a.rgb8, b.rgb8)
    assert np.array_equal(a.tri, b.tri) and np.array_equal(bits(a.t), bits(b.t)) and np.array_equal(bits(a.v), bits(b.v))
    assert np.array_equal(a.occ_tri, b.occ_tri) and np.array_equal(bits(a.rgb), bits(b.rgb))


def _with(s, **arrays):
    """the Scene s with some arrays replaced (same topology)"""
    return dataclasses.replace(s, **{k: np.array(v, np.float32) for k, v in arrays.items()})


def _fresh(renderer, s, **kw):
    rs = renderer.upload(s)
    try:
        return renderer.trace(rs, _cam(), W, H, debug=True, **kw)
    finally:
        rs.close()


def _moved_geometry(s, g, centre=(0.0, 1.3, 0.6)):
    """geometry g gathered into a cluster of triangles three times their size around centre (in view, between the floor
    and the lights): returns (first triangle, new vertices [n, 3, 3])"""
    a, b = int(s.geom_tri_offset[g]), int(s.geom_tri_offset[g + 1])
    v = s.tri_verts[a:b].astype(np.float64)
    c = v.mean(axis=1, keepdims=True)
    new = np.asarray(centre) + (c - c.mean(axis=0)) * 0.3 + (v - c) * 3.0
    return a, new.astype(np.float32)


def _render_modes(renderer, rs, **kw):
    return [renderer.trace(rs, _cam(), W, H, debug=True, rng_mode=0, seed=3, **m, **kw) for m in MODES]


def test_moved_geometry_hazard(renderer):
    """rows of the kept shadow tables and a kept tree would be stale: the moved triangles are hit and occlude after the
    update, and every mode and rng mode gives the fresh scene's frame"""
    from esctp1raytracer_b200 import RNG_EXPLICIT, RNG_HASH, hash_faceids, scenes

    s = scenes.soup_scene(20000, 40, 4, seed=5)
    g = 1 + s.n_lights  # the first geometry of the soup
    a, new = _moved_geometry(s, g)
    s2 = _with(s, tri_verts=np.concatenate([s.tri_verts[:a], new, s.tri_verts[a + len(new):]]))
    rs = renderer.upload(s)
    before = _render_modes(renderer, rs)  # builds the eye, shadow tables and the tree of the old geometry
    rs.update(tri_verts=new, first_tri=a)
    after = _render_modes(renderer, rs)
    assert not np.array_equal(before[0].rgb8, after[0].rgb8)
    moved = lambda x: (x >= a) & (x < a + len(new))
    assert moved(after[0].tri).sum() > 50 and moved(after[0].occ_tri).sum() > 50
    for m, f in zip(MODES, after):
        _same_frames(f, _fresh(renderer, s2, rng_mode=RNG_HASH, seed=3, **m))
    fid = hash_faceids(11, W, H, s.faces_per_light)
    _same_frames(renderer.trace(rs, _cam(), W, H, debug=True, rng_mode=RNG_EXPLICIT, faceid=fid),
                 _fresh(renderer, s2, rng_mode=RNG_EXPLICIT, faceid=fid))
    ex = renderer.trace(rs, _cam(), W, H, debug=True, rng_mode=RNG_HASH, seed=3, exhaustive_strict=True)
    assert ex.stats["filter_misses"] == 0 and ex.stats["pipeline_errors"] == 0
    _same_frames(ex, after[0])


def test_moved_light(renderer):
    from esctp1raytracer_b200 import scenes

    s = scenes.soup_scene(20000, 40, 4, seed=5)
    a, b = int(s.geom_tri_offset[1]), int(s.geom_tri_offset[2])  # light 0's quad
    new = s.tri_verts[a:b] + np.array([0.35, -0.25, 0.2], np.float32)
    s2 = _with(s, tri_verts=np.concatenate([s.tri_verts[:a], new, s.tri_verts[b:]]))
    rs = renderer.upload(s)
    before = _render_modes(renderer, rs)
    rs.update(tri_verts=new, first_tri=a)
    after = _render_modes(renderer, rs)
    assert not np.array_equal(before[0].occ_tri[:, 0], after[0].occ_tri[:, 0])  # light 0's shadows moved
    for m, f in zip(MODES, after):
        _same_frames(f, _fresh(renderer, s2, rng_mode=0, seed=3, **m))


def test_update_and_back_restores_the_frame(renderer):
    from esctp1raytracer_b200 import scenes

    s = scenes.soup_scene(20000, 40, 4, seed=7, n_spheres=20)
    rs = renderer.upload(s)
    before = _render_modes(renderer, rs)
    rng = np.random.default_rng(2)
    moved = (s.tri_verts + rng.normal(scale=0.05, size=s.tri_verts.shape)).astype(np.float32)
    rs.update(tri_verts=moved)
    mid = _render_modes(renderer, rs)
    for m, f in zip(MODES, mid):
        _same_frames(f, _fresh(renderer, _with(s, tri_verts=moved), rng_mode=0, seed=3, **m))
    rs.update(tri_verts=s.tri_verts)
    for f0, f in zip(before, _render_modes(renderer, rs)):
        _same_frames(f0, f)


def test_materials_spheres_normals(renderer):
    from esctp1raytracer_b200 import TracerError, scenes

    s = scenes.soup_scene(6000, 20, 2, seed=9, edge=(0.05, 0.2), with_normals=True, specular=True, n_spheres=30)
    rng = np.random.default_rng(4)
    mats = s.geom_material.copy()
    mats[1 + s.n_lights:, 3:9] = rng.uniform(0, 0.9, size=(s.n_geoms - 1 - s.n_lights, 6))
    sph = s.sphere_cr.copy()
    sph[:, :3] += rng.uniform(-0.3, 0.3, size=(len(sph), 3)).astype(np.float32)
    sph[:, 3] *= 3
    smat = s.sphere_material.copy()
    smat[:, 6:9] = 0.4
    a, n = 100, 2000
    nrm = s.tri_normals.copy()
    nrm[a:a + n] = -nrm[a:a + n]
    s2 = _with(s, geom_material=mats, sphere_cr=sph, sphere_material=smat, tri_normals=nrm)
    rs = renderer.upload(s)
    _render_modes(renderer, rs)
    rs.update(geom_material=mats, sphere_cr=sph)
    rs.update(sphere_material=smat, tri_normals=nrm[a:a + n], first_tri=a)
    for m, f in zip(MODES, _render_modes(renderer, rs)):
        _same_frames(f, _fresh(renderer, s2, rng_mode=0, seed=3, **m))
    plain = renderer.upload(scenes.soup_scene(6000, 20, 2, seed=9))
    with pytest.raises(TracerError, match="-1"):
        plain.update(tri_normals=nrm[:10])


def test_device_inputs_equal_host_inputs(renderer):
    import torch

    from esctp1raytracer_b200 import scenes

    s = scenes.soup_scene(20000, 40, 4, seed=5, n_spheres=10)
    a, new = _moved_geometry(s, 1 + s.n_lights)
    mats = s.geom_material.copy()
    mats[5:, 3:6] *= 0.5
    host = renderer.upload(s)
    dev = renderer.upload(s)
    _render_modes(renderer, host)
    _render_modes(renderer, dev)
    old = s.tri_verts[a:a + len(new)]
    delta = (new - old).astype(np.float32)
    want = (old + delta).astype(np.float32)  # what the device computes below: one float32 add per element
    host.update(tri_verts=want, first_tri=a, geom_material=mats)
    base, d = torch.from_numpy(old).cuda(), torch.from_numpy(delta).cuda()
    m = torch.from_numpy(mats).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(50_000_000)  # the side stream is busy for a while before it writes the vertices
        t = base + d
    dev.update(tri_verts=t, first_tri=a, geom_material=m, stream=side.cuda_stream)  # no host synchronise before
    for fh, fd in zip(_render_modes(renderer, host), _render_modes(renderer, dev)):
        _same_frames(fh, fd)
    # the interface has no stream entry: the legacy default stream (torch's), behind work queued there
    dev.update(tri_verts=torch.from_numpy(s.tri_verts).cuda())
    host.update(tri_verts=s.tri_verts)
    for fh, fd in zip(_render_modes(renderer, host), _render_modes(renderer, dev)):
        _same_frames(fh, fd)


def test_seeded_bands_after_update(renderer):
    from esctp1raytracer_b200 import RNG_MT19937, scenes

    s = scenes.soup_scene(20000, 40, 4, seed=5)
    a, new = _moved_geometry(s, 2 + s.n_lights)
    s2 = _with(s, tri_verts=np.concatenate([s.tri_verts[:a], new, s.tri_verts[a + len(new):]]))
    rs = renderer.upload(s)
    renderer.trace(rs, _cam(), W, H, rng_mode=RNG_MT19937, seed=9)
    rs.update(tri_verts=new, first_tri=a)
    for m in MODES:
        whole = _fresh(renderer, s2, rng_mode=RNG_MT19937, seed=9, **m)
        frame_rows = (whole.tri.reshape(H, W) >= 0).sum(1).astype(np.int32)

        def hook(row_hits):
            row_hits[:] = frame_rows

        rgb8 = np.zeros_like(whole.rgb8)
        for bi in range(3):
            rows = [pr for pr in range(H) if (pr // 8) % 3 == bi]
            part = renderer.trace(rs, _cam(), W, H, rng_mode=RNG_MT19937, seed=9, bands=(8, bi, 3), debug=True,
                                  row_hits_exchange=hook, **m)
            assert np.array_equal(part.tri.reshape(len(rows), W), whole.tri.reshape(H, W)[rows])
            rgb8[rows] = part.rgb8
        assert np.array_equal(rgb8, whole.rgb8)


def test_non_resident_tables(renderer, monkeypatch):
    from esctp1raytracer_b200 import scenes

    monkeypatch.setenv("TRACER_TABLE_SLOTS", "1")  # one light vertex's tables at a time: rebuilt every frame
    s = scenes.soup_scene(20000, 40, 4, seed=5)
    a, new = _moved_geometry(s, 1 + s.n_lights)
    b0, b1 = int(s.geom_tri_offset[2]), int(s.geom_tri_offset[3])
    lnew = s.tri_verts[b0:b1] + np.array([-0.2, -0.1, 0.1], np.float32)
    v2 = s.tri_verts.copy()
    v2[a:a + len(new)], v2[b0:b1] = new, lnew
    rs = renderer.upload(s)
    renderer.trace(rs, _cam(), W, H, rng_mode=0, seed=3)
    rs.update(tri_verts=new, first_tri=a)
    rs.update(tri_verts=lnew, first_tri=b0)
    f = renderer.trace(rs, _cam(), W, H, debug=True, rng_mode=0, seed=3)
    _same_frames(f, _fresh(renderer, _with(s, tri_verts=v2), rng_mode=0, seed=3))


def test_refused_updates_change_nothing(renderer):
    import torch

    from esctp1raytracer_b200 import TracerError, _lib, scenes

    s = scenes.soup_scene(20000, 40, 4, seed=5)
    rs = renderer.upload(s)
    before = _render_modes(renderer, rs)
    lib = renderer.lib
    a, new = _moved_geometry(s, 1 + s.n_lights)

    def raw(**fields):
        u = _lib.SceneUpdate()
        u.struct_size = C.sizeof(u)
        for k, v in fields.items():
            setattr(u, k, v)
        return lib.tracer_cuda_scene_update(rs.handle, C.byref(u))

    with pytest.raises(TracerError, match="-1"):
        rs.update(tri_verts=new, first_tri=s.n_tris - 5)  # past the end
    with pytest.raises(TracerError, match="-1"):
        rs.update(tri_verts=new, first_tri=-1)
    assert raw(tri_first=a, tri_count=len(new)) == -1  # a count without data
    assert raw(struct_size=8, tri_first=a, tri_count=len(new), tri_verts=new.ctypes.data) == -1
    assert raw(data_is_device=1, tri_first=a, tri_count=len(new), tri_verts=new.ctypes.data) == -1  # host memory
    assert raw(data_is_device=1, geom_material=s.geom_material.ctypes.data) == -1
    if torch.cuda.device_count() >= 2:
        with pytest.raises(TracerError, match="-1"):
            rs.update(tri_verts=torch.from_numpy(new).to("cuda:1"), first_tri=a)
    assert raw() == 0  # nothing to do
    for f0, f in zip(before, _render_modes(renderer, rs)):
        _same_frames(f0, f)


def _bbox(lib, rs):
    out = (C.c_double * 6)()
    lib.tracer__scene_bbox.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    assert lib.tracer__scene_bbox(rs.handle, out) == 0
    return np.array(out[:], np.float64)


def _bbox_loop(s):
    """the host loop scene creation used to run: std::min / std::max in order, vertices then spheres"""
    lo, hi = [1e300] * 3, [-1e300] * 3
    items = [(x, x) for x in s.tri_verts.reshape(-1, 3).astype(np.float64)]
    items += [(c - r, c + r) for c, r in zip(s.sphere_cr[:, :3].astype(np.float64), np.abs(s.sphere_cr[:, 3].astype(np.float64)))]
    for xl, xh in items:
        for k in range(3):
            lo[k] = xl[k] if xl[k] < lo[k] else lo[k]
            hi[k] = xh[k] if hi[k] < xh[k] else hi[k]
    return np.array(lo + hi, np.float64)


def test_bounding_box(renderer):
    from esctp1raytracer_b200 import Scene, scenes

    s = scenes.soup_scene(300, 6, 1, n_spheres=4, seed=2)
    v = s.tri_verts.copy()
    v[20, 1, 0] = np.nan  # skipped
    v[21, 2, 2] = np.inf  # counts
    v[22, 0, 1] = -0.0    # equal to the floor's +0.0, which comes first: +0.0 stays
    s = _with(s, tri_verts=v)
    rs = renderer.upload(s)
    got, want = _bbox(renderer.lib, rs), _bbox_loop(s)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (got, want)
    assert got[5] == np.inf and got[1] == 0.0 and not np.signbit(got[1])
    v2 = v.copy()
    v2[0, :, 1] = -0.0  # now the first zero is -0.0
    v2[23] = [[np.nan, np.nan, np.nan], [-np.inf, 5.0, np.nan], [1.0, 1.0, 1.0]]
    sph = s.sphere_cr.copy()
    sph[2] = [0.0, 9.0, 0.0, -2.5]  # |r| is used
    sph[3] = [np.nan, 1.5, np.inf, 1.0]  # x -+ r = NaN, z +- r = inf
    s2 = _with(s, tri_verts=v2, sphere_cr=sph)
    rs.update(tri_verts=v2[:24], sphere_cr=sph)
    got, want = _bbox(renderer.lib, rs), _bbox_loop(s2)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (got, want)
    assert np.signbit(got[1]) and got[0] == -np.inf and got[4] == 11.5
    rs2 = renderer.upload(s2)
    assert np.array_equal(_bbox(renderer.lib, rs2).view(np.uint64), want.view(np.uint64))
    empty = renderer.upload(Scene(np.array([0]), np.zeros((0, 3, 3)), np.zeros((0, 13)), np.zeros(0)))
    assert list(_bbox(renderer.lib, empty)) == [1e300] * 3 + [-1e300] * 3
    big = scenes.soup_scene(200000, 100, 4, n_spheres=100, seed=8)
    vb = big.tri_verts.copy()
    vb[::997, 1, 2] = np.nan
    big = _with(big, tri_verts=vb)
    b = _bbox(renderer.lib, renderer.upload(big))
    vv = vb.reshape(-1, 3).astype(np.float64)
    c, r = big.sphere_cr[:, :3].astype(np.float64), np.abs(big.sphere_cr[:, 3:].astype(np.float64))
    assert np.array_equal(b, np.concatenate([np.fmin(np.nanmin(vv, 0), (c - r).min(0)), np.fmax(np.nanmax(vv, 0), (c + r).max(0))]))


def test_full_size_c4_one_geometry(renderer):
    from esctp1raytracer_b200 import RNG_HASH, Camera, scenes

    Wf, Hf = 3840, 2160
    s = scenes.soup_scene(1_000_000, 1000, 4, n_spheres=1000, seed=42)
    cam = Camera.for_frame(EYE, LOOK, Wf, Hf)
    a, new = _moved_geometry(s, 500)  # about 1000 triangles
    v2 = s.tri_verts.copy()
    v2[a:a + len(new)] = new
    rs = renderer.upload(s)
    renderer.trace(rs, cam, Wf, Hf, rng_mode=RNG_HASH, seed=42)
    rs.update(tri_verts=new, first_tri=a)
    got = renderer.trace(rs, cam, Wf, Hf, rng_mode=RNG_HASH, seed=42).rgb8
    rs.close()
    fresh = renderer.upload(_with(s, tri_verts=v2))
    want = renderer.trace(fresh, cam, Wf, Hf, rng_mode=RNG_HASH, seed=42).rgb8
    assert hashlib.sha256(got.tobytes()).hexdigest() == hashlib.sha256(want.tobytes()).hexdigest()


def test_multi_gpu_update(renderer):
    import torch

    from esctp1raytracer_b200 import RNG_HASH, MultiRenderer, Renderer, scenes

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two or more GPUs")
    s = scenes.soup_scene(20000, 40, 4, seed=5)
    a, new = _moved_geometry(s, 1 + s.n_lights)
    mats = s.geom_material.copy()
    mats[6:, 3:6] *= 0.25
    s2 = _with(s, tri_verts=np.concatenate([s.tri_verts[:a], new, s.tri_verts[a + len(new):]]), geom_material=mats)
    Wm, Hm = 200, 150
    cam = _cam(Wm, Hm)
    r1 = Renderer(0)
    want = r1.trace(r1.upload(s2), cam, Wm, Hm, rng_mode=RNG_HASH, seed=3).rgb8
    m = MultiRenderer(n)
    for source in ("host", "device"):
        ms = m.upload(s)
        m.trace(ms, cam, Wm, Hm, rng_mode=RNG_HASH, seed=3)
        if source == "host":
            ms.update(tri_verts=new, first_tri=a, geom_material=mats)
        else:
            ms.update(tri_verts=torch.from_numpy(new).to("cuda:0"), first_tri=a, geom_material=torch.from_numpy(mats).to("cuda:0"))
        for kw in (dict(), dict(bundle_cull=1), dict(bvh=True)):
            assert np.array_equal(m.trace(ms, cam, Wm, Hm, rng_mode=RNG_HASH, seed=3, **kw).rgb8, want), (source, kw)
        ms.close()
    Renderer(0)  # back to one GPU
