"""CPU checks of the HOT span rows (csrc/sweep.cuh: hot_row, hot_terms, hot_pass; the rows build_origin_table stores and
the default sweeps' hot loop reads) through the library's host build of the same source (tracer__hot_row_pass: no GPU).

The tables store span_rows' row with both constants of every bound shifted by -(1 - delta), rounded up.  A thread then forms
A = min3(lower bounds, clamp), B = min3(upper bounds, clamp) and tests |2 S p + (A - B)| <= A + B.  The frame stays the same
when that test drops no pair the saturating span test passes (and hence none the reference accepts):

* rays aimed as tests/test_filter_rows.py aims them at random, needle-shaped, coplanar-with-the-origin and light-owned
  triangles: every pair the restated reference accepts passes the hot loop's shared-q test (both q modes) and the
  candidate path's per-ray test with the ray's own q;
* rays on and a few ulps around both ends of each interval, rows in any position and with steep q slopes: every pair the
  saturating form passes passes the hot test, every pair span_pass passes passes the per-ray test, and a row stored with
  delta = 0 loses some of them, so the margin is needed;
* on random rays the hot test passes about as many pairs as the interval form it replaces;
* padding rows stay never-candidate and rows without bounds always-candidate.
"""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

from esctp1raytracer_b200 import _lib
from test_filter_interval import PMAX, S, edge_rays, iv, primary_cases  # noqa: F401
from test_filter_rows import F32, aim_points, face_param, flt, qbar_form, random_triangle, shadow_setup  # noqa: F401

F32P = C.POINTER(C.c_float)
U = 2.0 ** -24


def fptr(a):
    return a.ctypes.data_as(F32P)


@pytest.fixture(scope="module")
def hot(flt):
    lib = _lib.load()
    lib.tracer__hot_row_pass.argtypes = [F32P, C.c_int, F32P, F32P, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_ubyte), F32P]
    lib.tracer__hot_row_pass.restype = None
    lib.tracer__hot_consts.argtypes = [F32P]
    lib.tracer__hot_consts.restype = None
    consts = np.zeros(3, F32)
    lib.tracer__hot_consts(fptr(consts))

    class Hot:
        CLAMP, DELTA, QD_SCALE = (float(c) for c in consts)
        rows, accepts, camera = flt.rows, flt.accepts, flt.camera

        @staticmethod
        def passes(row8, p, q, qbar, qdelta=-1.0, delta=None):
            """bit 0 hot loop (shared q), bit 1 per-ray hot test (own q), bit 2 saturating form (shared q), bit 3 span_pass
            (own q), bit 4 the interval form it replaces (shared q)"""
            p = np.ascontiguousarray(p, F32)
            q = np.ascontiguousarray(np.broadcast_to(np.asarray(q, F32), p.shape), F32)
            out = np.zeros(len(p), np.uint8)
            row8 = np.ascontiguousarray(row8, F32)
            lib.tracer__hot_row_pass(fptr(row8), len(p), fptr(p), fptr(q), float(qbar), float(qdelta),
                                     float(Hot.DELTA if delta is None else delta), out.ctypes.data_as(C.POINTER(C.c_ubyte)), None)
            return out

        @staticmethod
        def stored(row8, delta=None):
            hot8 = np.zeros(8, F32)
            out = np.zeros(1, np.uint8)
            lib.tracer__hot_row_pass(fptr(np.ascontiguousarray(row8, F32)), 0, fptr(np.zeros(1, F32)), fptr(np.zeros(1, F32)), 0.0, -1.0,
                                     float(Hot.DELTA if delta is None else delta), out.ctypes.data_as(C.POINTER(C.c_ubyte)), fptr(hot8))
            return hot8

    return Hot


def test_constants_match_the_derivation(hot):
    assert hot.CLAMP == float(S) * PMAX + 1.0
    assert hot.DELTA == pytest.approx(8 * 1.1920929e-7 * hot.CLAMP, rel=1e-6)
    Q = hot.CLAMP + 2
    assert hot.DELTA >= (4.2 * U * Q + 3.5 * U) + 3 * U * hot.CLAMP + U * U * hot.CLAMP  # the bound derived at HOT_DELTA
    assert hot.CLAMP >= float(S) * PMAX + hot.DELTA
    assert hot.QD_SCALE == 1.0 + 2.0 ** -20


def test_shift_is_rounded_up_exactly(hot):
    """C' is the least float >= C - (1 - delta), for constants of every magnitude and sign"""
    rng = np.random.default_rng(30)
    mags = np.concatenate([10.0 ** rng.uniform(-30, 30, 3000), rng.uniform(0, 4, 500), [0.0, 1.0, 1e30, 2.0 ** 24, 2.0 ** 25 + 2]])
    c = (mags * rng.choice([-1.0, 1.0], len(mags))).astype(F32)
    s = Fraction(1) - Fraction(float(F32(hot.DELTA)))
    n_checked = 0
    for i in range(0, len(c) - 1, 2):
        row = np.array([0.5, c[i], -0.25, c[i + 1], 0.0, 1e30, 0.0, 1e30], F32)
        h = hot.stored(row)
        for k in (1, 3):
            exact = Fraction(float(row[k])) - s
            assert Fraction(float(h[k])) >= exact and Fraction(float(np.nextafter(h[k], F32(-np.inf)))) < exact, (row[k], h[k])
            n_checked += 1
        assert h[0] == row[0] and h[2] == row[2]  # q coefficients unchanged
    assert n_checked > 3000


def test_primary_rays_the_reference_accepts_pass_the_hot_tests(hot):
    rng = np.random.default_rng(31)
    n_acc = 0
    for rows, p, q, acc in primary_cases(hot, rng, 200):
        row8 = rows[12:20]
        for i in np.nonzero(acc)[0]:
            # MODE_SHAREDQ: the ray among others of the same image row; the candidate path with the same q
            pp = np.concatenate([p[i:i + 1], rng.uniform(0, 1, 3).astype(F32)])
            res = hot.passes(row8, pp, q[i], q[i])
            assert res[0] & 3 == 3, (rows, p[i], q[i])
        for i in np.nonzero(acc)[0][:6]:  # jittered samples: mean q + |B| * spread (MODE_QBAR)
            qbar, qdelta = qbar_form(rng, q[i])
            assert hot.passes(row8, p[i:i + 1], q[i], qbar, qdelta)[0] & 3 == 3, (rows, p[i], q[i], qbar, qdelta)
        n_acc += int(acc.sum())
    assert n_acc > 5000


def test_shadow_rays_the_reference_accepts_pass_the_hot_tests(hot):
    rng = np.random.default_rng(32)
    n_acc = n_own = 0
    for it in range(200):
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
        X = aim_points(rng, tri, 200)
        alpha = np.where(rng.uniform(size=len(X)) < 0.9, 1 + 10 ** rng.uniform(-4, 0.5, len(X)), rng.uniform(0.2, 0.999, len(X)))
        hit = (lv[None, :] + (X - lv[None, :]) * alpha[:, None]).astype(F32)
        hit = hit[np.linalg.norm(hit - lv[None, :], axis=1) > 1e-6]
        d, t, face, p, q, ln = shadow_setup(hit, lv)
        acc = hot.accepts(hit, d, tri, t)
        for f in np.unique(face):
            rows = hot.rows(tri, *face_param(lv, int(f)), float(ln.max()) * 1.5)
            for i in np.nonzero((face == f) & acc)[0]:
                qbar, qdelta = qbar_form(rng, q[i])  # the shadow sweeps' shared q-term; the candidate path: own q
                assert hot.passes(rows[12:20], p[i:i + 1], q[i], qbar, qdelta)[0] & 3 == 3, (it, f, tri, lv, hit[i], qbar, qdelta)
        n_acc += int(acc.sum())
    assert n_acc > 4000 and n_own >= 15


def synthetic_rows(rng, n):
    """rows in any position of the frame, one lower and one upper bound (second slots open), shallow and steep q slopes"""
    for k in range(n):
        ql = F32(rng.uniform(-1, 1))
        lo_p, hi_p = np.sort(rng.uniform(-PMAX, PMAX, 2))
        if rng.uniform() < 0.2:
            hi_p = lo_p + rng.uniform(0, 1e-4)
        steep = k % 3 == 0  # nearly horizontal edges: |B| up to ~1e11 row units, where |B| * qdelta dominates
        bl, bu = ((10 ** rng.uniform(0, 6.2) if steep else 0.3) * rng.normal() for _ in range(2))
        row8 = np.zeros(8, F32)
        row8[0:4] = [F32(-S * bl), F32(1 - S * (lo_p - bl * ql)), 0, F32(1e30)]
        row8[4:8] = [F32(S * bu), F32(1 + S * (hi_p - bu * ql)), 0, F32(1e30)]
        yield row8, ql


def test_margin_covers_the_saturating_form_and_is_needed(hot, iv):
    """every pair the saturating form passes passes the hot loop's test, every pair span_pass passes the per-ray test;
    stored with delta = 0 some do not"""
    rng = np.random.default_rng(33)
    n_sat = n_own = lost_without_margin = 0

    def check(row8, qi, qdelta):
        nonlocal n_sat, n_own, lost_without_margin
        rows20 = np.concatenate([np.zeros(12, F32), row8])
        pe = edge_rays(rows20, qi, qdelta, rng)
        res = hot.passes(row8, pe, qi, qi, qdelta)
        sat, own = (res & 4) != 0, (res & 8) != 0
        # the saturating form here is tracer__interval_pass' bit 1, bit for bit
        assert np.array_equal(sat, (iv.passes(rows20, pe, qi, qdelta) & 2) != 0)
        assert np.all(res[sat] & 1), (row8, qi, qdelta, pe[sat & ((res & 1) == 0)])
        assert np.all(res[own] & 2), (row8, qi, pe[own & ((res & 2) == 0)])
        bare = hot.passes(row8, pe, qi, qi, qdelta, delta=0.0)
        lost_without_margin += int(np.sum(sat & ((bare & 1) == 0))) + int(np.sum(own & ((bare & 2) == 0)))
        n_sat += int(sat.sum())
        n_own += int(own.sum())

    for rows, p, q, acc in primary_cases(hot, rng, 120):
        for qi, qdelta in [(q[0], -1.0), qbar_form(rng, q[0])]:
            check(rows[12:20], qi, qdelta)
    for row8, ql in synthetic_rows(rng, 3000):
        for qi, qdelta in [(ql, -1.0), qbar_form(rng, ql)]:
            check(row8, qi, qdelta)
    assert n_sat > 50000 and n_own > 50000
    assert lost_without_margin > 0, "delta = 0 should lose pairs at the interval ends"


def test_candidate_count_close_to_the_interval_form(hot):
    rng = np.random.default_rng(34)
    n_hot = n_iv = 0
    for rows, p, q, acc in primary_cases(hot, rng, 150):
        pr = rng.uniform(0, 1, 512).astype(F32)
        res = hot.passes(rows[12:20], np.concatenate([p, pr]), q[0], q[0])
        n_hot += int(np.sum(res & 1 != 0))
        n_iv += int(np.sum(res & 16 != 0))
    print(f"pairs passing: hot form {n_hot}, interval form {n_iv} ({n_hot / n_iv - 1:+.4%})")
    assert n_iv > 1000 and n_hot <= 1.001 * n_iv


def test_padding_and_always_candidate_rows(hot):
    p = np.linspace(-PMAX, PMAX, 257, dtype=F32)
    pad = np.array([0, -1e30, 0, -1e30, 0, 1e30, 0, 1e30], F32)  # build_origin_table's / build_allcand_table's padding
    allc = np.array([0, 1e30, 0, 1e30, 0, 1e30, 0, 1e30], F32)  # no bound at all: always candidate
    assert np.array_equal(hot.stored(pad), pad) and np.array_equal(hot.stored(allc), allc)  # the shift leaves 1e30 as it is
    for q, qdelta in [(0.5, -1.0), (0.5, 1e-6), (-1.0, 1e-4)]:
        assert not np.any(hot.passes(pad, p, q, q, qdelta) & 3)
        assert np.all(hot.passes(allc, p, q, q, qdelta) & 3 == 3)
    one_sided = np.array([0, 1 - 0.25 * 65536, 0, 1e30, 0, 1e30, 0, 1e30], F32)  # p >= 0.25 only
    res = hot.passes(one_sided, p, 0.0, 0.0)
    assert np.array_equal((res & 4) != 0, p >= 0.25) and np.all(res[p >= 0.25] & 3 == 3)
