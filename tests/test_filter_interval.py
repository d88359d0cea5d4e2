"""CPU checks of the interval form of the span test (csrc/sweep.cuh: span_interval, interval_pass, the hot loop of the
default sweeps) through the library's host build of the same source (tracer__interval_pass: no GPU needed).

The hot loop decides per (thread, triangle) whether any of the thread's rays may hit the triangle, as min_r |S p_r - c| <= h
with (c, h) the centre and widened half width of the span row's interval of S p.  The candidate path re-checks flagged
triangles ray by ray with the unchanged per-ray test, so the frame stays the same exactly when the interval form never drops
a pair that the saturating form (x = sat(S p + ax), y = sat(ay - S p) both 1) passes, and hence none the reference accepts:

* rays aimed as tests/test_filter_rows.py aims them (primary rays on the image plane, shadow rays on the cube faces of a
  light vertex, with the shared-q form of the shadow sweeps) at the interiors, edges and vertices of random, needle-shaped,
  coplanar-with-the-origin and light-owned triangles: every pair the restated reference accepts passes the interval form;
* rays placed on and a few ulps around both ends of each interval: every pair the saturating form passes passes the
  interval form, and a build without the margin (delta = 0, clamp box S * PMAX) fails that check, so the margin is needed;
* on random rays the interval form passes only a few percent more pairs than the saturating form.
"""
import ctypes as C

import numpy as np
import pytest

from esctp1raytracer_b200 import _lib
from test_filter_rows import FLT_MAX, F32, aim_points, f32_normalize, face_param, flt, qbar_form, random_triangle, shadow_setup  # noqa: F401

F32P = C.POINTER(C.c_float)
S = F32(65536.0)
PMAX = 1.0625


def fptr(a):
    return a.ctypes.data_as(F32P)


@pytest.fixture(scope="module")
def iv(flt):
    lib = _lib.load()
    lib.tracer__interval_pass.argtypes = [F32P, C.c_int, F32P, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_ubyte)]
    lib.tracer__interval_pass.restype = None
    lib.tracer__interval_consts.argtypes = [F32P]
    lib.tracer__interval_consts.restype = None
    consts = np.zeros(2, F32)
    lib.tracer__interval_consts(fptr(consts))
    box, delta = float(consts[0]), float(consts[1])

    class Iv:
        BOX, DELTA = box, delta
        rows, accepts, camera = flt.rows, flt.accepts, flt.camera

        @staticmethod
        def passes(rows20, p, q, qdelta=-1.0, box=box, delta=delta):
            """bit 0 interval form, bit 1 saturating form, bit 2 per-ray span_pass (q as the rays' own q)"""
            p = np.ascontiguousarray(p, F32)
            out = np.zeros(len(p), np.uint8)
            row8 = np.ascontiguousarray(rows20[12:20], F32)
            lib.tracer__interval_pass(fptr(row8), len(p), fptr(p), float(q), float(qdelta), float(box), float(delta),
                                      out.ctypes.data_as(C.POINTER(C.c_ubyte)))
            return out

    return Iv


def test_constants_match_the_derivation(iv):
    assert iv.BOX == float(S) * PMAX + 1.0
    assert iv.DELTA == pytest.approx(8 * 1.1920929e-7 * iv.BOX, rel=1e-6)
    assert iv.DELTA * 3840 < float(S) / 100  # far below a pixel of a 3840-wide frame


def primary_cases(iv, rng, n_tri):
    """(rows, p, q, accepted) per triangle, rays built as test_filter_rows builds primary rays"""
    for it in range(n_tri):
        eye = np.array([0, 1, 3], F32) + rng.normal(size=3).astype(F32) * F32(0.3)
        look = np.array([0, 1, 0], F32) + rng.normal(size=3).astype(F32) * F32(0.2)
        o, llc, hor, ver = iv.camera(eye, look, F32(rng.choice([3840 / 2160, 1.0])))
        U, V, Wv = hor.astype(np.float64), ver.astype(np.float64), llc.astype(np.float64) - o.astype(np.float64)
        dmax = max(np.linalg.norm(Wv + a * U + b * V) for a in (0, 1) for b in (0, 1))
        s, t = rng.uniform(0.05, 0.95, 2)
        dist = 10 ** rng.uniform(-0.5, 1.3)
        centre = o + (Wv + s * U + t * V) / np.linalg.norm(Wv + s * U + t * V) * dist
        tri = random_triangle(rng, centre, dist * 10 ** rng.uniform(-3.5, -0.3), needle=it % 5 == 0)
        if it % 13 == 0:  # the eye (nearly) in the triangle's plane
            nrm = np.cross(tri[1] - tri[0], tri[2] - tri[0]).astype(np.float64)
            nrm /= max(np.linalg.norm(nrm), 1e-30)
            tri = (tri + (nrm * np.dot(o - tri[0], nrm) * (1 - rng.choice([0.0, 1e-7, 1e-5])))[None, :]).astype(F32)
        rows = iv.rows(tri, o, U, V, Wv, dmax, 0.0)
        X = aim_points(rng, tri, 200)
        M = np.stack([np.broadcast_to(U, X.shape), np.broadcast_to(V, X.shape), -(X - o)], axis=2)
        try:
            sol = np.linalg.solve(M, np.broadcast_to(-Wv, X.shape)[..., None])[..., 0]
        except np.linalg.LinAlgError:
            continue
        p, q = sol[:, 0].astype(F32), sol[:, 1].astype(F32)
        keep = (sol[:, 2] > 0) & (p >= 0) & (p <= 1) & (q >= 0) & (q <= 1)
        p, q = p[keep], q[keep]
        if len(p) == 0:
            continue
        p = np.clip(np.nextafter(p, F32(rng.choice([-1, 2]))), 0, 1).astype(F32)
        d = ((llc[None, :] + (hor[None, :] * p[:, None]).astype(F32)).astype(F32) + (ver[None, :] * q[:, None]).astype(F32)).astype(F32)
        d = f32_normalize((d - o[None, :]).astype(F32))
        yield rows, p, q, iv.accepts(o, d, tri, FLT_MAX)


def test_primary_rays_the_reference_accepts_pass_the_interval_form(iv):
    rng = np.random.default_rng(21)
    n_acc = 0
    for rows, p, q, acc in primary_cases(iv, rng, 200):
        for i in np.nonzero(acc)[0]:
            # MODE_SHAREDQ: the thread's rays share the ray's q exactly; the ray among others of the same image row
            res = iv.passes(rows, np.concatenate([p[i:i + 1], rng.uniform(0, 1, 3).astype(F32)]), q[i])
            assert res[0] & 1, (rows, p[i], q[i])
        for i in np.nonzero(acc)[0][:6]:  # jittered samples: mean q + |B| * spread (MODE_QBAR)
            qbar, qdelta = qbar_form(rng, q[i])
            assert iv.passes(rows, p[i:i + 1], qbar, qdelta)[0] & 1, (rows, p[i], q[i], qbar, qdelta)
        n_acc += int(acc.sum())
    assert n_acc > 5000


def test_shadow_rays_the_reference_accepts_pass_the_interval_form(iv):
    rng = np.random.default_rng(22)
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
        acc = iv.accepts(hit, d, tri, t)
        for f in np.unique(face):
            rows = iv.rows(tri, *face_param(lv, int(f)), float(ln.max()) * 1.5)
            for i in np.nonzero((face == f) & acc)[0]:
                qbar, qdelta = qbar_form(rng, q[i])  # the shadow sweeps' shared q-term
                assert iv.passes(rows, p[i:i + 1], qbar, qdelta)[0] & 1, (it, f, tri, lv, hit[i], qbar, qdelta)
        n_acc += int(acc.sum())
    assert n_acc > 4000 and n_own >= 15


def edge_rays(rows, q, qdelta, rng):
    """p at and a few ulps around both ends of the saturating form's interval (and at the box edges)"""
    lo, hi = rows[12:16].astype(np.float64), rows[16:20].astype(np.float64)
    qq = np.float64(q)
    ax = min(qq * lo[0] + lo[1], qq * lo[2] + lo[3]) - (abs(lo[0]) + abs(lo[2])) * max(qdelta, 0)
    ay = min(qq * hi[0] + hi[1], qq * hi[2] + hi[3]) - (abs(hi[0]) + abs(hi[2])) * max(qdelta, 0)
    ends = np.array([(1 - ax) / float(S), (ay - 1) / float(S), -PMAX, PMAX, 0.0])
    ends = ends[np.isfinite(ends) & (np.abs(ends) <= PMAX)]
    p = np.repeat(ends, 41).astype(F32)
    k = np.tile(np.arange(-20, 21), len(ends))
    p = p.view(np.int32) + np.sign(p).astype(np.int32) * k.astype(np.int32)
    p = np.clip(p.view(F32), -PMAX, PMAX).astype(F32)
    return np.concatenate([p, rng.uniform(-PMAX, PMAX, 16).astype(F32)])


def test_margin_covers_the_saturating_form_and_is_needed(iv):
    """every pair the saturating form passes passes the interval form; without the margin some do not"""
    rng = np.random.default_rng(23)
    n_sat = lost_without_margin = 0
    for rows, p, q, acc in primary_cases(iv, rng, 120):
        for qi, qdelta in [(q[0], -1.0), qbar_form(rng, q[0])]:
            pe = edge_rays(rows, qi, qdelta, rng)
            res = iv.passes(rows, pe, qi, qdelta)
            sat = (res & 2) != 0
            assert np.all(res[sat] & 1), (rows, qi, qdelta, pe[sat & ((res & 1) == 0)])
            bare = iv.passes(rows, pe, qi, qdelta, box=float(S) * PMAX, delta=0.0)
            lost_without_margin += int(np.sum(sat & ((bare & 1) == 0)))
            n_sat += int(sat.sum())
    # rows in any position of the frame, at the interval ends exactly
    for _ in range(3000):
        ql = F32(rng.uniform(0, 1))
        lo_p, hi_p = np.sort(rng.uniform(-PMAX, PMAX, 2))
        if rng.uniform() < 0.2:
            hi_p = lo_p + rng.uniform(0, 1e-4)
        rows = np.zeros(20, F32)
        # lower bound p >= lo_p (+ q slope), upper bound p <= hi_p; the second slot of each side open
        bl, bu = rng.normal() * 0.3, rng.normal() * 0.3
        rows[12:16] = [F32(-S * bl), F32(1 - S * (lo_p - bl * ql)), 0, F32(1e30)]
        rows[16:20] = [F32(S * bu), F32(1 + S * (hi_p - bu * ql)), 0, F32(1e30)]
        for qi, qdelta in [(ql, -1.0), qbar_form(rng, ql)]:
            pe = edge_rays(rows, qi, qdelta, rng)
            res = iv.passes(rows, pe, qi, qdelta)
            sat = (res & 2) != 0
            assert np.all(res[sat] & 1), (rows, qi, qdelta, pe[sat & ((res & 1) == 0)])
            bare = iv.passes(rows, pe, qi, qdelta, box=float(S) * PMAX, delta=0.0)
            lost_without_margin += int(np.sum(sat & ((bare & 1) == 0)))
            n_sat += int(sat.sum())
    assert n_sat > 50000
    assert lost_without_margin > 0, "delta = 0 without the clamp margin should lose pairs at the interval ends"


def test_padding_open_and_always_candidate_rows(iv):
    p = np.linspace(-PMAX, PMAX, 257, dtype=F32)
    pad = np.array([0] * 12 + [0, -1e30, 0, -1e30, 0, 1e30, 0, 1e30], F32)  # build_origin_table's padding rows
    allc = np.array([0] * 12 + [0, 1e30, 0, 1e30, 0, 1e30, 0, 1e30], F32)  # no bound at all: always candidate
    for q, qdelta in [(0.5, -1.0), (0.5, 1e-6), (-1.0, 1e-4)]:
        assert not np.any(iv.passes(pad, p, q, qdelta) & 3)
        assert np.all(iv.passes(allc, p, q, qdelta) & 3 == 3)
    one_sided = np.array([0] * 12 + [0, 1 - 0.25 * 65536, 0, 1e30, 0, 1e30, 0, 1e30], F32)  # p >= 0.25 only
    res = iv.passes(one_sided, p, 0.0)
    assert np.array_equal((res & 2) != 0, p >= 0.25) and np.all(res[p >= 0.25] & 1)


def test_candidate_count_close_to_the_saturating_form(iv):
    rng = np.random.default_rng(24)
    n_iv = n_sat = 0
    for rows, p, q, acc in primary_cases(iv, rng, 150):
        pr = rng.uniform(0, 1, 512).astype(F32)
        res = iv.passes(rows, np.concatenate([p, pr]), q[0])
        n_iv += int(np.sum(res & 1 != 0))
        n_sat += int(np.sum(res & 2 != 0))
    print(f"pairs passing: interval form {n_iv}, saturating form {n_sat} ({n_iv / n_sat - 1:+.3%})")
    assert n_sat > 1000 and n_sat <= n_iv <= 1.03 * n_sat
