"""CPU checks of the shadow sweeps' MEAN-q SEGMENT verdict (csrc/sweep.cuh: hot_terms_qbar, then segment_pass) through the
library's host build of the same source (tracer__segment_pass_qbar: no GPU).

A shadow thread holds R rays of one (p, q) cell of its ray group.  They share one (nc2, h2): the hot row's bounds at the
thread's mean q, widened by |B| * qdelta with qdelta >= max |q_r - qbar| (shadow_item's formula).  The verdict tests
fl(pmin2 + nc2) <= h2 and fl(pmax2 + nc2) >= -h2 on the least and greatest 2 S p of the thread, so it is, exactly,

    not (every ray's sum > h2)  and  not (every ray's sum < -h2),

which holds whenever one ray passes the per-ray test at qbar, and that test passes every pair the reference accepts.
These tests check the identity and the implications on:

* shadow rays aimed at random, needle-shaped, coplanar-with-the-light and light-owned triangles that the restated reference
  accepts, placed in cells of 32 rays with q spreads from 0 to 1e-2, in any order;
* rays on and a few ulps around both ends of each row's interval, on rows with shallow and steep q slopes;
* padding rows (never) and rows without bounds (always);

and that a verdict taken from the cell's first and last rays, or one with qdelta = 0 over a spread of q, fails them.
"""
import ctypes as C

import numpy as np
import pytest

from esctp1raytracer_b200 import _lib
from test_filter_interval import PMAX, S  # noqa: F401
from test_filter_rows import F32, aim_points, face_param, flt, random_triangle, shadow_setup  # noqa: F401
from test_hot_rows import hot, synthetic_rows  # noqa: F401

F32P = C.POINTER(C.c_float)
S2 = F32(2.0 * float(S))
R = 32
SPREADS = (0.0, 1e-6, 1e-4, 1e-3, 1e-2)


def fptr(a):
    return a.ctypes.data_as(F32P)


@pytest.fixture(scope="module")
def segq():
    lib = _lib.load()
    lib.tracer__segment_pass_qbar.argtypes = [F32P, C.c_int, F32P, F32P, C.c_float, C.c_float, C.POINTER(C.c_ubyte), F32P]
    lib.tracer__segment_pass_qbar.restype = None

    def run(row8, p, q, qbar=None, qdelta=None):
        """-> (verdict, OR of the per-ray tests at qbar, OR with each ray's own q, nc2, h2); qbar/qdelta default to
        shadow_item's over all of q"""
        p, q = np.ascontiguousarray(p, F32), np.ascontiguousarray(q, F32)
        if qbar is None:
            qbar, qdelta = cell_qbar(q)
        out, terms = np.zeros(3, np.uint8), np.zeros(2, F32)
        lib.tracer__segment_pass_qbar(fptr(np.ascontiguousarray(row8, F32)), len(p), fptr(p), fptr(q), float(qbar), float(qdelta),
                                      out.ctypes.data_as(C.POINTER(C.c_ubyte)), fptr(terms))
        return bool(out[0]), bool(out[1]), bool(out[2]), terms[0], terms[1]

    return run


def cell_qbar(q):
    """shadow_item (kernels.cuh): qbar and qdelta of a thread's q values, float32 throughout"""
    qmin, qmax = F32(np.min(q)), F32(np.max(q))
    qbar = F32(F32(0.5) * F32(qmin + qmax))
    qdelta = F32(F32(max(F32(qmax - qbar), F32(qbar - qmin))) * F32(1.0001) + F32(2.4e-7) * F32(abs(qbar) + F32(1)))
    return qbar, qdelta


def sums(p, nc2):
    return (np.asarray(p, F32) * S2).astype(F32) + nc2  # float32: one RN rounding per operation


class Cells:
    def __init__(self, segq):
        self.segq, self.items = segq, []
        self.n_any = self.n_own = self.n_extra = 0

    def check(self, row8, p, q):
        v, any_ray, own, nc2, h2 = self.segq(row8, p, q)
        e = sums(p, nc2)
        assert any_ray == bool(np.any(np.abs(e) <= h2))
        assert v == (not np.all(e > h2) and not np.all(e < -h2)), (row8, p, q, nc2, h2)
        assert v or not any_ray, (row8, p, q)
        self.n_any += any_ray
        self.n_own += own
        self.n_extra += v and not any_ray
        self.items.append((row8, np.array(p, F32), np.array(q, F32), nc2, h2, own, v))
        return v, any_ray, own


def cell(rng, p0, q0, spread):
    """ray (p0, q0) among 31 others of a cell: p within a few triangle widths, q within +-spread, in random order"""
    n = R - 1
    p = (p0 + rng.uniform(-0.02, 0.02, n)).astype(F32)
    q = (q0 + spread * rng.uniform(-1, 1, n)).astype(F32)
    if rng.uniform() < 0.2:  # a short list's tail: the last entry duplicated
        p[-5:], q[-5:] = p[-6], q[-6]
    idx = rng.permutation(R)
    return np.concatenate([[F32(p0)], p]).astype(F32)[idx], np.concatenate([[F32(q0)], q]).astype(F32)[idx]


def test_shadow_rays_the_reference_accepts_pass_in_cells(segq, hot):
    rng = np.random.default_rng(81)
    cells = Cells(segq)
    n_acc = n_own = 0
    for it in range(160):
        lv = (np.array([0, 1.9, 0]) + rng.normal(size=3) * 0.5).astype(F32)
        dist = 10 ** rng.uniform(-1.0, 0.8)
        dirn = rng.normal(size=3)
        dirn /= np.linalg.norm(dirn)
        tri = random_triangle(rng, lv + dirn * dist, dist * 10 ** rng.uniform(-3.0, -0.2), needle=it % 5 == 0)
        if it % 11 == 0:  # light-owned: the light vertex is a vertex of the triangle
            tri[rng.integers(0, 3)] = lv
            n_own += 1
        elif it % 11 == 1:  # the light vertex in the triangle's plane
            nrm = np.cross(tri[1] - tri[0], tri[2] - tri[0]).astype(np.float64)
            nrm /= max(np.linalg.norm(nrm), 1e-30)
            tri = (tri + (nrm * np.dot(lv - tri[0], nrm))[None, :]).astype(F32)
        X = aim_points(rng, tri, 120)
        alpha = np.where(rng.uniform(size=len(X)) < 0.9, 1 + 10 ** rng.uniform(-4, 0.5, len(X)), rng.uniform(0.2, 0.999, len(X)))
        hit = (lv[None, :] + (X - lv[None, :]) * alpha[:, None]).astype(F32)
        hit = hit[np.linalg.norm(hit - lv[None, :], axis=1) > 1e-6]
        d, t, face, p, q, ln = shadow_setup(hit, lv)
        acc = hot.accepts(hit, d, tri, t)
        for f in np.unique(face):
            row8 = hot.rows(tri, *face_param(lv, int(f)), float(ln.max()) * 1.5)[12:20]
            for i in np.nonzero((face == f) & acc)[0][:12]:
                for spread in SPREADS:
                    pp, qq = cell(rng, p[i], q[i], spread)
                    v, any_ray, own = cells.check(row8, pp, qq)
                    assert v and any_ray and own, (it, f, tri, lv, hit[i], spread)
                n_acc += 1
    print(f"accepted rays {n_acc}, cells {len(cells.items)}, verdict set with no ray passing at qbar {cells.n_extra}")
    assert n_acc > 1500 and n_own >= 10


def hot_ends(nc2, h2):
    return [(-float(h2) - float(nc2)) / float(S2), (float(h2) - float(nc2)) / float(S2)]


def test_rays_around_the_interval_ends(segq):
    rng = np.random.default_rng(82)
    cells = Cells(segq)
    n_single = 0
    for row8, ql in synthetic_rows(rng, 500):
        spread = float(rng.choice(SPREADS))
        q = (ql + spread * rng.uniform(-1, 1, R)).astype(F32)
        _, _, _, nc2, h2 = segq(row8, np.zeros(R, F32), q)
        if not h2 > 0:
            continue
        for end in hot_ends(nc2, h2):
            if abs(end) > PMAX:
                continue
            pe = (np.repeat(F32(end), 15).view(np.int32) + np.arange(-7, 8, dtype=np.int32)).view(F32)
            out = F32(1.0 if end > float(-nc2) / float(S2) else -1.0)
            step = F32(2e-4)
            for x in pe:
                outside = (x + out * step * np.arange(1, R, dtype=F32)).astype(F32)
                inside = (x - out * step * np.arange(1, R, dtype=F32)).astype(F32)
                for pp in (np.concatenate([[x], outside]), rng.permutation(np.concatenate([[x], outside])),
                           np.concatenate([inside[: R // 2], [x], outside[: R // 2 - 1]])):
                    _, any_ray, _ = cells.check(row8, pp, q)
                    n_single += any_ray
    print(f"cells {len(cells.items)}, with a ray passing at qbar {cells.n_any}")
    assert n_single > 2000 and cells.n_any > 3000


def test_wrong_verdicts_fail(segq, hot):
    """a verdict from the cell's first and last rays, or one computed with qdelta = 0 over a spread of q, loses pairs"""
    rng = np.random.default_rng(83)
    ends_lost = qd0_lost = 0
    for row8, ql in synthetic_rows(rng, 600):
        for spread in (1e-4, 1e-3, 1e-2):
            q = (ql + spread * rng.uniform(-1, 1, R)).astype(F32)
            _, _, _, nc2, h2 = segq(row8, np.zeros(R, F32), q)
            if not h2 > 0:
                continue
            mid = F32(-float(nc2) / float(S2))
            p = np.sort((mid + rng.uniform(-0.03, 0.03, R)).astype(F32))
            p = np.concatenate([p[R // 2:], p[: R // 2]])  # first and last rays are not the extremes
            v, any_ray, own, nc2, h2 = segq(row8, p, q)
            e = sums(p, nc2)
            if any_ray and (e[0] > h2 or -e[-1] > h2):
                ends_lost += 1
            qbar, _ = cell_qbar(q)
            v0, _, _, _, _ = segq(row8, p, q, qbar, 0.0)
            if own and not v0:
                qd0_lost += 1
    assert ends_lost > 0, "a verdict from the first and last rays should lose some cells"
    assert qd0_lost > 0, "a verdict without the |B| * qdelta widening should lose some cells"


def test_padding_and_always_candidate_rows(segq):
    rng = np.random.default_rng(84)
    pad = np.array([0, -1e30, 0, -1e30, 0, 1e30, 0, 1e30], F32)
    allc = np.array([0, 1e30, 0, 1e30, 0, 1e30, 0, 1e30], F32)
    for _ in range(60):
        p = rng.uniform(-PMAX, PMAX, R).astype(F32)
        q = (rng.uniform(-1, 1) + rng.choice(SPREADS) * rng.uniform(-1, 1, R)).astype(F32)
        assert segq(pad, p, q)[:3] == (False, False, False)
        assert segq(allc, p, q)[:3] == (True, True, True)
    extreme = np.array([-PMAX, PMAX], F32)
    assert segq(pad, extreme, np.zeros(2, F32))[0] is False and segq(allc, extreme, np.zeros(2, F32))[0] is True
