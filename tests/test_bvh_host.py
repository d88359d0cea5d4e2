"""CPU checks of the optional BVH mode (csrc/bvh.cuh) through the library's host build of the same source
(tracer__bvh_build_host, tracer__bvh_query_host: no GPU needed).

BVH mode is exact when the traversal never skips a (ray, triangle) pair the reference's test accepts.  Here:

* the tree: every finite triangle in exactly one leaf, boxes that contain their children, correct smallest index and
  largest sigma per child, triangles that are not finite (or too large for the margin argument) on the always-test list;
* the traversal against brute force (the strict test on every triangle, in index order), closest hit and first occluder,
  bit for bit, on ~10^5 rays built in float as the device builds them: primary rays through the image plane and shadow
  rays from on-surface points towards a light vertex, aimed at interiors, edges and vertices, needle triangles,
  triangles coplanar with the origin, axis-aligned rays (+-0 direction components) and grazing rays;
* the margins are needed: the same traversal with m = 0 and no sigma terms loses pairs on this set.
"""
import ctypes as C

import numpy as np
import pytest

from esctp1raytracer_b200 import _lib
from test_filter_rows import EPS, F32, FLT_MAX, aim_points, f32_normalize, flt, random_triangle, shadow_setup  # noqa: F401

F32P = C.POINTER(C.c_float)
I32P = C.POINTER(C.c_int32)


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


@pytest.fixture(scope="module")
def bh():
    lib = _lib.load()
    lib.tracer__bvh_build_host.argtypes = [C.c_int, F32P, F32P, I32P, I32P, I32P]
    lib.tracer__bvh_build_host.restype = C.c_int
    lib.tracer__bvh_query_host.argtypes = [C.c_int, F32P, F32P, C.c_int, C.c_int, I32P, C.c_int, C.c_int, F32P, F32P, F32P,
                                           C.c_int, C.c_int, C.c_float, C.c_float, I32P, F32P, C.POINTER(C.c_longlong)]
    lib.tracer__bvh_query_host.restype = None
    lib.tracer__bvh_margin.argtypes = [C.c_double, C.c_double]
    lib.tracer__bvh_margin.restype = C.c_float

    class Bvh:
        @staticmethod
        def build(verts):
            v = np.ascontiguousarray(verts, F32).reshape(-1, 9)
            n = len(v)
            nodes = np.zeros((max(n - 1, 1), 20), F32)
            always = np.zeros(max(n, 1), np.int32)
            root_leaf, n_always = C.c_int32(), C.c_int32()
            n_in = lib.tracer__bvh_build_host(n, _p(v, C.c_float), _p(nodes, C.c_float), C.byref(root_leaf),
                                              _p(always, C.c_int32), C.byref(n_always))
            return dict(verts=v, nodes=nodes, n_in=n_in, root_leaf=root_leaf.value, always=always[:n_always.value].copy())

        @staticmethod
        def margin(verts, o, lmax):
            v = np.asarray(verts, np.float64).reshape(-1, 3)
            v = v[np.all(np.isfinite(v), axis=1)]
            ext = max(float(np.abs(v).max()) if len(v) else 0.0, float(np.abs(o).max()))
            return lib.tracer__bvh_margin(ext, lmax)

        @staticmethod
        def query(tree, o, d, t, mode, brute, m, dscale=1.0):
            o, d = np.ascontiguousarray(o, F32).reshape(-1, 3), np.ascontiguousarray(d, F32).reshape(-1, 3)
            o = np.ascontiguousarray(np.broadcast_to(o, d.shape), F32)
            t = np.ascontiguousarray(np.broadcast_to(np.asarray(t, F32), (len(d),)), F32)
            idx, tout, tests = np.zeros(len(d), np.int32), np.zeros(len(d), F32), C.c_longlong()
            v = tree["verts"]
            lib.tracer__bvh_query_host(len(v), _p(v, C.c_float), _p(tree["nodes"], C.c_float), tree["n_in"], tree["root_leaf"],
                                       _p(tree["always"], C.c_int32), len(tree["always"]), len(d), _p(o, C.c_float),
                                       _p(d, C.c_float), _p(t, C.c_float), mode, int(brute), m, dscale,
                                       _p(idx, C.c_int32), _p(tout, C.c_float), C.byref(tests))
            return idx, tout.view(np.uint32), tests.value

    return Bvh


def sigma_of(v):
    v = v.reshape(-1, 3, 3).astype(F32)
    e1, e2 = (v[:, 1] - v[:, 0]).astype(F32), (v[:, 2] - v[:, 0]).astype(F32)
    return np.linalg.norm(e1.astype(np.float64), axis=1) * np.linalg.norm(e2.astype(np.float64), axis=1)


def check_tree(tree):
    v = tree["verts"].reshape(-1, 3, 3)
    n = len(v)
    finite = np.all(np.isfinite(v.reshape(n, 9)), axis=1)
    with np.errstate(all="ignore"):
        sig = sigma_of(v)
    in_tree = finite & np.isfinite(sig) & (sig < 0.125)
    assert tree["n_in"] == int(in_tree.sum())
    assert sorted(tree["always"].tolist()) == tree["always"].tolist() == np.nonzero(~in_tree)[0].tolist()
    nodes = tree["nodes"]
    child, mn = nodes[:, 16:18].view(np.int32), nodes[:, 18:20].view(np.int32)
    seen = []

    def box_of_tri(i):
        return v[i].min(axis=0), v[i].max(axis=0)

    def visit(node):
        """-> (lo, hi, min index, max sigma) of the subtree, checking what the node stores about each child"""
        out = []
        for c in range(2):
            ch = int(child[node, c])
            lo_s, hi_s, s_s = nodes[node, 8 * c:8 * c + 3], nodes[node, 8 * c + 4:8 * c + 7], nodes[node, 8 * c + 3]
            if ch < 0:
                tri = ~ch
                seen.append(tri)
                lo, hi = box_of_tri(tri)
                sub = (lo, hi, tri, sig[tri])
            else:
                sub = visit(ch)
            assert np.all(lo_s <= sub[0]) and np.all(hi_s >= sub[1]), (node, c)  # the box contains the child
            assert np.array_equal(lo_s, sub[0]) and np.array_equal(hi_s, sub[1])  # ... and is its exact union
            assert mn[node, c] == sub[2]
            assert s_s >= sub[3] and s_s <= sub[3] * (1 + 1e-5) + 1e-30
            out.append(sub)
        return (np.minimum(out[0][0], out[1][0]), np.maximum(out[0][1], out[1][1]), min(out[0][2], out[1][2]),
                max(out[0][3], out[1][3]))

    if tree["n_in"] >= 2:
        visit(0)
    elif tree["n_in"] == 1:
        seen.append(tree["root_leaf"])
    assert sorted(seen) == np.nonzero(in_tree)[0].tolist()  # every tree triangle in exactly one leaf


def scenes(rng):
    out = {}
    c = rng.uniform(-1, 1, (3000, 3))  # small triangles, as in the soup scenes: the tree prunes
    out["random"] = (c[:, None, :] + rng.normal(size=(3000, 3, 3)) * 0.008).astype(F32)
    c = rng.uniform(-1, 1, (300, 3))  # medium triangles: the sigma terms dilate the boxes much more
    out["medium"] = (c[:, None, :] + rng.normal(size=(300, 3, 3)) * 0.05).astype(F32)
    out["identical"] = np.repeat(random_triangle(rng, np.zeros(3), 0.1)[None], 64, axis=0)
    g = []
    for i in range(8):  # coplanar, axis-aligned: a tiled floor y = 0 and a wall x = 0.5 (zero-thickness boxes)
        for j in range(8):
            x0, z0 = -1 + i * 0.25, -1 + j * 0.25
            g += [[[x0, 0, z0], [x0 + 0.25, 0, z0], [x0 + 0.25, 0, z0 + 0.25]], [[x0, 0, z0], [x0 + 0.25, 0, z0 + 0.25], [x0, 0, z0 + 0.25]]]
            g += [[[0.5, x0 + 1, z0], [0.5, x0 + 1.25, z0], [0.5, x0 + 1.25, z0 + 0.25]]]
    out["coplanar"] = np.array(g, F32)
    out["one"] = random_triangle(rng, np.zeros(3), 0.2)[None]
    needles = np.array([random_triangle(rng, rng.uniform(-1, 1, 3), 0.08, needle=True) for _ in range(100)], F32)
    bad = np.array([[[np.nan, 0, 0], [1, 0, 0], [0, 1, 0]], [[np.inf, 0, 0], [1, 0, 0], [0, 1, 0]],
                    [[1e30, 0, -1e30], [0, 1e30, -1e30], [-1e30, -1e30, -1e30]], [[-3, -0.5, -3], [3, -0.5, -3], [0, -0.5, 3]]], F32)
    out["needles_and_outsiders"] = np.concatenate([needles, bad[:3], out["medium"][:100], bad[3:]]).astype(F32)
    return out


def test_tree_invariants(bh):
    rng = np.random.default_rng(31)
    for name, v in scenes(rng).items():
        with np.errstate(all="ignore"):
            check_tree(bh.build(v))
    assert bh.build(np.zeros((0, 3, 3), F32))["n_in"] == 0


def primary_rays(rng, v, n_aim):
    """camera rays in float through aim points on the triangles (test_filter_rows' construction) + random ones"""
    from test_filter_rows import F32 as _F  # noqa: F401
    from esctp1raytracer_b200 import Camera

    eye = (np.array([0, 1, 3]) + rng.normal(size=3) * 0.3).astype(F32)
    cam = np.asarray(Camera(eye, (0, 0.3, 0), (0, 1, 0), 60.0, 16 / 9).as_array(), F32).reshape(12)
    o, llc, hor, ver = cam[0:3], cam[3:6], cam[6:9], cam[9:12]
    U, V, Wv = hor.astype(np.float64), ver.astype(np.float64), llc.astype(np.float64) - o.astype(np.float64)
    fin = np.all(np.isfinite(v.reshape(len(v), 9)), axis=1) & (np.abs(v.reshape(len(v), 9)).max(axis=1) < 100)
    idx = np.nonzero(fin)[0]
    X = np.concatenate([aim_points(rng, v[i].astype(np.float64), n_aim) for i in rng.choice(idx, min(len(idx), 120))])
    M = np.stack([np.broadcast_to(U, X.shape), np.broadcast_to(V, X.shape), -(X - o)], axis=2)
    sol = np.linalg.solve(M, np.broadcast_to(-Wv, X.shape)[..., None])[..., 0]
    p, q = sol[:, 0], sol[:, 1]
    keep = (sol[:, 2] > 0) & (p > -0.5) & (p < 1.5) & (q > -0.5) & (q < 1.5)
    p, q = np.concatenate([p[keep], rng.uniform(0, 1, 500)]).astype(F32), np.concatenate([q[keep], rng.uniform(0, 1, 500)]).astype(F32)
    p = np.nextafter(p, F32(rng.choice([-1, 2]))).astype(F32)
    d = ((llc[None, :] + (hor[None, :] * p[:, None]).astype(F32)).astype(F32) + (ver[None, :] * q[:, None]).astype(F32)).astype(F32)
    return o, f32_normalize((d - o[None, :]).astype(F32))


def shadow_rays(rng, v, n_aim, lv):
    """on-surface origins (points of the triangles, in float) towards a light vertex, as light_step_kernel sets them up"""
    fin = np.all(np.isfinite(v.reshape(len(v), 9)), axis=1) & (np.abs(v.reshape(len(v), 9)).max(axis=1) < 100)
    idx = np.nonzero(fin)[0]
    hit = np.concatenate([aim_points(rng, v[i].astype(np.float64), n_aim) for i in rng.choice(idx, min(len(idx), 120))]).astype(F32)
    hit = hit[np.linalg.norm(hit - lv[None, :], axis=1) > 1e-4]
    d, t, face, p, q, ln = shadow_setup(hit, lv)
    return hit, d, t


def special_rays(rng, v):
    """axis-aligned rays (+-0 components), rays grazing a triangle's plane, rays from a triangle's own vertex"""
    o, d = [], []
    fin = np.nonzero(np.all(np.isfinite(v.reshape(len(v), 9)), axis=1) & (np.abs(v.reshape(len(v), 9)).max(axis=1) < 100))[0]
    for i in rng.choice(fin, min(len(fin), 60)):
        X = aim_points(rng, v[i].astype(np.float64), 20).astype(F32)
        for a in range(3):  # axis-aligned rays onto the aim points, both senses, with -0 / +0 elsewhere
            dd = np.zeros((len(X), 3), F32)
            dd[:, a] = rng.choice([-1.0, 1.0])
            dd[:, (a + 1) % 3] = rng.choice([0.0, -0.0])
            oo = X.copy()
            oo[:, a] -= dd[:, a] * F32(2.5)
            o.append(oo), d.append(dd)
        e1, e2 = (v[i, 1] - v[i, 0]).astype(np.float64), (v[i, 2] - v[i, 0]).astype(np.float64)
        nrm = np.cross(e1, e2)
        nrm /= max(np.linalg.norm(nrm), 1e-30)
        inplane = rng.normal(size=(len(X), 3))
        inplane -= (inplane @ nrm)[:, None] * nrm[None, :]
        inplane += nrm[None, :] * rng.choice([0.0, 1e-7, -1e-6, 1e-4], (len(X), 1))  # grazing
        dd = f32_normalize(inplane.astype(F32))
        o.append((X - dd * F32(1.7)).astype(F32)), d.append(dd)
        o.append(np.repeat(v[i, rng.integers(0, 3)][None], len(X), 0)), d.append(f32_normalize(rng.normal(size=(len(X), 3)).astype(F32)))
    return np.concatenate(o).astype(F32), np.concatenate(d).astype(F32)


def run_case(bh, tree, o, d, t, mode, m, dscale=1.0):
    ib, tb, nb = bh.query(tree, o, d, t, mode, True, m)
    it, tt, nt = bh.query(tree, o, d, t, mode, False, m, dscale)
    return ib, tb, it, tt, nb, nt


def all_cases(bh, rng):
    for name, v in scenes(rng).items():
        with np.errstate(all="ignore"):
            tree = bh.build(v)
        lv = (np.array([0, 1.9, 0]) + rng.normal(size=3) * 0.3).astype(F32)
        o, d = primary_rays(rng, v, 60)
        yield name, "primary", tree, o, d, FLT_MAX, 0, bh.margin(v, o, 10.0)
        o, d = special_rays(rng, v)
        yield name, "special", tree, o, d, FLT_MAX, 0, bh.margin(v, o, 10.0)
        yield name, "special-occ", tree, o, d, F32(3.0), 1, bh.margin(v, o, 10.0)
        o, d, t = shadow_rays(rng, v, 60, lv)
        yield name, "shadow", tree, o, d, t, 1, bh.margin(v, o, 10.0)


def test_traversal_matches_brute_force(bh, flt):
    rng = np.random.default_rng(32)
    n_rays = n_hits = n_tests_tree = n_tests_brute = 0
    spot = 0
    for name, kind, tree, o, d, t, mode, m in all_cases(bh, rng):
        with np.errstate(all="ignore"):
            ib, tb, it, tt, nb, nt = run_case(bh, tree, o, d, t, mode, m)
        bad = np.nonzero((ib != it) | ((ib >= 0) & (tb != tt)))[0]
        assert len(bad) == 0, (name, kind, bad[:5], ib[bad[:5]], it[bad[:5]])
        n_rays += len(d)
        n_hits += int((ib >= 0).sum())
        n_tests_tree += nt
        n_tests_brute += nb
        # spot-check the brute-force answers against the restated reference
        oo = np.ascontiguousarray(np.broadcast_to(o.reshape(-1, 3), d.shape), F32)
        tt0 = np.broadcast_to(np.asarray(t, F32), (len(d),))
        for r in rng.choice(np.nonzero(ib >= 0)[0], min(8, int((ib >= 0).sum())), replace=False) if (ib >= 0).any() else []:
            tri = tree["verts"][ib[r]].reshape(3, 3)
            assert flt.accepts(oo[r], d[r:r + 1], tri, FLT_MAX if mode == 0 else tt0[r])[0], (name, kind, r)
            spot += 1
    print(f"{n_rays} rays, {n_hits} hits/occluders, strict tests: tree {n_tests_tree}, brute force {n_tests_brute}")
    assert n_rays > 50000 and n_hits > 10000 and spot > 50
    assert n_tests_tree < n_tests_brute


def test_margins_are_needed(bh):
    """with m = 0 and no sigma terms in the box test, the same traversal loses pairs the strict test accepts"""
    rng = np.random.default_rng(32)
    lost = 0
    for name, kind, tree, o, d, t, mode, m in all_cases(bh, rng):
        with np.errstate(all="ignore"):
            ib, tb, it, tt, nb, nt = run_case(bh, tree, o, d, t, mode, 0.0, dscale=0.0)
        lost += int(np.sum((ib != it) | ((ib >= 0) & (tb != tt))))
    print("pairs lost without the margins:", lost)
    assert lost > 0, "m = 0 and no sigma terms should lose pairs on this set"
