"""CPU checks of the closest-hit sweep's SEGMENT verdict (csrc/sweep.cuh: segment_pass, eval_segment) through the library's
host build of the same source (tracer__segment_pass: no GPU).

A closest-hit thread holds R pixels of one image row, so its rays share q and hence (nc2, h2).  The per-ray loop passes a
triangle when some ray has |fl(2 S p + nc2)| <= h2; the segment verdict tests fl(pmin2 + nc2) <= h2 and
fl(pmax2 + nc2) >= -h2 on the least and greatest 2 S p of the thread.  As round-to-nearest addition is monotone and pmin2,
pmax2 are themselves rays of the thread, the verdict is, exactly,

    not (every ray's sum > h2)  and  not (every ray's sum < -h2),

which holds whenever some ray passes.  These tests check that identity and that implication on:

* rays aimed at random, needle-shaped and coplanar-with-the-eye triangles that the restated reference accepts, placed among
  other pixels of their row in any order;
* runs of 64 pixels of a 3840-wide row (p = w / (W - 1)), unsorted, with the duplicated edge pixels a frame-edge thread holds;
* rays on and a few ulps around both ends of each row's hot interval;
* intervals that fall between two neighbouring pixels of a run, where the verdict may pass with no ray passing (counted);
* padding rows (never) and rows without bounds (always);

and that a verdict taken from the run's first and last rays, or one that drops either side, fails them.
"""
import ctypes as C

import numpy as np
import pytest

from esctp1raytracer_b200 import _lib
from test_filter_interval import PMAX, S, primary_cases  # noqa: F401
from test_filter_rows import F32, flt  # noqa: F401
from test_hot_rows import hot, synthetic_rows  # noqa: F401

F32P = C.POINTER(C.c_float)
S2 = F32(2.0 * float(S))
W_FRAME, R = 3840, 64


def fptr(a):
    return a.ctypes.data_as(F32P)


@pytest.fixture(scope="module")
def seg():
    lib = _lib.load()
    lib.tracer__segment_pass.argtypes = [F32P, C.c_int, F32P, C.c_float, C.POINTER(C.c_ubyte), F32P]
    lib.tracer__segment_pass.restype = None

    def run(row8, p, q):
        """-> (segment verdict, OR of the per-ray hot tests, nc2, h2)"""
        p = np.ascontiguousarray(p, F32)
        out, terms = np.zeros(2, np.uint8), np.zeros(2, F32)
        lib.tracer__segment_pass(fptr(np.ascontiguousarray(row8, F32)), len(p), fptr(p), float(q), out.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                 fptr(terms))
        return bool(out[0]), bool(out[1]), terms[0], terms[1]

    return run


def sums(p, nc2):
    return (np.asarray(p, F32) * S2).astype(F32) + nc2  # float32 throughout: one RN rounding per operation


def required(p, nc2, h2):
    e = sums(p, nc2)
    return not np.all(e > h2) and not np.all(e < -h2)


# deliberately wrong verdicts (the tests below must reject each of them)
def ends_verdict(p, nc2, h2):  # the run's first and last rays, not its least and greatest
    e0, e1 = sums(p[:1], nc2)[0], sums(p[-1:], nc2)[0]
    return not e0 > h2 and not -e1 > h2


def lower_side_only(p, nc2, h2):
    return not sums([np.min(p)], nc2)[0] > h2


def upper_side_only(p, nc2, h2):
    return not -sums([np.max(p)], nc2)[0] > h2


def pixel_p(w):
    return (np.asarray(w, F32) / F32(W_FRAME - 1)).astype(F32)  # pixel_st: p = w / (W - 1), one RN division


def pixel_run(x0):
    """the 64 rays of a thread starting at pixel x0, edge pixels duplicated past the frame's edge"""
    return pixel_p(np.minimum(np.arange(x0, x0 + R), W_FRAME - 1))


class Cases:
    """(row8, p, q) runs checked against the verdict, with the totals the tests report"""

    def __init__(self, seg):
        self.seg, self.items = seg, []
        self.n_any = self.n_extra = 0

    def check(self, row8, p, q):
        v, any_ray, nc2, h2 = self.seg(row8, p, q)
        assert any_ray == bool(np.any(np.abs(sums(p, nc2)) <= h2))  # the hook's per-ray OR is hot_pass's
        assert v == required(p, nc2, h2), (row8, q, p, nc2, h2)
        assert v or not any_ray, (row8, q, p, nc2, h2)
        self.n_any += any_ray
        self.n_extra += v and not any_ray
        self.items.append((np.array(p, F32), nc2, h2, any_ray, v))
        return v, any_ray

    def rejects(self, verdict):
        """some run on which `verdict` breaks what the segment verdict must satisfy"""
        return any(verdict(p, nc2, h2) != v or (any_ray and not verdict(p, nc2, h2)) for p, nc2, h2, any_ray, v in self.items)


def around(p0, rng, n_grid=R - 1):
    """p0 among pixels of its row near it, in random order, with some duplicates"""
    w0 = int(np.clip(np.rint(float(p0) * (W_FRAME - 1)), 0, W_FRAME - 1))
    x0 = int(rng.integers(max(0, w0 - n_grid), w0 + 1))
    run = pixel_p(np.minimum(np.arange(x0, x0 + n_grid), W_FRAME - 1))
    return rng.permutation(np.concatenate([run, [p0]]).astype(F32))


def test_aimed_rays_the_reference_accepts_pass_the_segment_verdict(seg, hot):
    rng = np.random.default_rng(71)
    cases = Cases(seg)
    n_acc = 0
    for rows, p, q, acc in primary_cases(hot, rng, 200):
        row8 = rows[12:20]
        for i in np.nonzero(acc)[0][:20]:
            for pp in (around(p[i], rng), p[i:i + 1], np.repeat(p[i], 3)):
                v, any_ray = cases.check(row8, pp, q[i])
                assert any_ray and v, (rows, p[i], q[i])
            n_acc += 1
        for _ in range(4):  # runs of pixels of the ray's row anywhere in the frame
            cases.check(row8, rng.permutation(pixel_run(int(rng.integers(0, W_FRAME)))), q[0])
    assert n_acc > 1000 and cases.n_any > 3000


def hot_ends(nc2, h2):
    """the p at which 2 S p + nc2 = -h2 and = h2 (float64: the ulp sweep below covers the rounding)"""
    return [(-float(h2) - float(nc2)) / float(S2), (float(h2) - float(nc2)) / float(S2)]


def test_rays_around_the_interval_ends_and_unsorted_runs(seg, hot):
    rng = np.random.default_rng(72)
    cases = Cases(seg)
    n_single = 0
    rowsets = [(rows[12:20], q[0]) for rows, p, q, acc in primary_cases(hot, rng, 60)] + list(synthetic_rows(rng, 600))
    for row8, q in rowsets:
        _, _, nc2, h2 = seg(row8, np.zeros(1, F32), q)
        if not h2 > 0:
            continue
        for end in hot_ends(nc2, h2):
            if abs(end) > PMAX:
                continue
            pe = np.repeat(F32(end), 21).view(np.int32) + np.sign(F32(end)).astype(np.int32) * np.arange(-10, 11, dtype=np.int32)
            pe = pe.view(F32)
            for x in pe:
                # one ray at the end, the others all past it on the outside, inside, or both; in any order
                step = F32(1.0 / (W_FRAME - 1))
                out = F32(np.sign(end - float(-nc2) / float(S2)) or 1.0)
                outside = (x + out * step * np.arange(1, 8, dtype=F32)).astype(F32)
                inside = (x - out * step * np.arange(1, 8, dtype=F32)).astype(F32)
                for pp in ([x], np.concatenate([outside, [x]]), np.concatenate([[x], outside, outside[:2]]),
                           rng.permutation(np.concatenate([outside, [x], inside])), np.concatenate([inside[::-1], [x]])):
                    _, any_ray = cases.check(row8, np.asarray(pp, F32), q)
                    n_single += any_ray
        # 64-pixel runs, ascending, descending and shuffled, and frame-edge runs with duplicated edge pixels
        for x0 in (int(rng.integers(0, W_FRAME - R)), W_FRAME - int(rng.integers(1, R))):
            run = pixel_run(x0)
            for pp in (run, run[::-1], rng.permutation(run)):
                cases.check(row8, pp, q)
    print(f"runs {len(cases.items)}, with a passing ray {cases.n_any}, verdict set with none passing {cases.n_extra}")
    assert n_single > 2000 and cases.n_any > 5000
    assert cases.rejects(ends_verdict), "a verdict from the first and last rays should fail these runs"
    assert cases.rejects(lower_side_only) and cases.rejects(upper_side_only), "a one-sided verdict should fail these runs"


def test_intervals_between_neighbouring_pixels(seg):
    """a triangle whose interval lies between two neighbouring rays of a run: no ray passes, the verdict may"""
    rng = np.random.default_rng(73)
    cases = Cases(seg)
    n_between = 0
    for _ in range(2000):
        x0 = int(rng.integers(0, W_FRAME - R))
        run = pixel_run(x0)
        k = int(rng.integers(0, R - 1))
        a, b = float(run[k]), float(run[k + 1])
        lo_p, hi_p = np.sort(rng.uniform(a + 0.05 * (b - a), b - 0.05 * (b - a), 2))
        ql = F32(rng.uniform(0, 1))
        bl, bu = 0.3 * rng.normal(), 0.3 * rng.normal()
        row8 = np.array([-S * bl, 1 - S * (lo_p - bl * ql), 0, 1e30, S * bu, 1 + S * (hi_p - bu * ql), 0, 1e30], F32)
        for pp in (run, rng.permutation(run)):
            v, any_ray = cases.check(row8, pp, ql)
            assert not any_ray
            n_between += v
    print(f"intervals between two neighbouring pixels: verdict set in {n_between} of {len(cases.items)} runs")
    assert n_between == len(cases.items)  # the run's rays lie on both sides of every such interval


def test_padding_and_always_candidate_rows(seg):
    rng = np.random.default_rng(74)
    pad = np.array([0, -1e30, 0, -1e30, 0, 1e30, 0, 1e30], F32)
    allc = np.array([0, 1e30, 0, 1e30, 0, 1e30, 0, 1e30], F32)
    cases = Cases(seg)
    for x0 in list(rng.integers(0, W_FRAME, 50)) + [0, W_FRAME - 1]:
        run = rng.permutation(pixel_run(int(x0)))
        for q in (0.0, 0.5, 1.0):
            assert cases.check(pad, run, q) == (False, False)
            assert cases.check(allc, run, q) == (True, True)
    extreme = np.array([-PMAX, PMAX], F32)
    assert cases.check(pad, extreme, 0.5) == (False, False) and cases.check(allc, extreme, 0.5) == (True, True)
    assert cases.rejects(lower_side_only), "dropping the upper side lets padding rows through"
