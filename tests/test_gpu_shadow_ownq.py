"""Shadow sweeps that rebuild a flagged triangle's pairs with each ray's own q, one ray per lane (sweep.cuh, sweep_table),
over rays ordered in square (p, q) cells (stripe_key_kernel).  Tall cells (stripes of 16384 entries, a whole group at
these sizes) give the same debug outputs as the oracle and bundle-cull mode, in exhaustive mode, in band shares, with
seeded faceIDs and in a crop window, and the pairs queued for the strict test no longer depend on the order: the same
within a few percent at stripe lengths 1, 4096 and the default."""
import re

import pytest

import test_gpu_shadow_cells as cells
from test_gpu_shadow_cells import renderer, stripe  # noqa: F401  (fixtures)
from test_gpu_shadow_lanes import _cases, _no_misses

pytestmark = pytest.mark.gpu

TALL = ("16384",)


@pytest.mark.parametrize("case", [0, 1, 6])
def test_tall_cells_equal_the_oracle_and_bundle_cull(renderer, restated, stripe, case, monkeypatch):  # noqa: F811
    monkeypatch.setattr(cells, "STRIPES", TALL)
    cells.test_cells_equal_the_oracle_and_bundle_cull(renderer, restated, stripe, case)


def test_tall_cells_seeded_faceids_and_crop(renderer, stripe, monkeypatch):  # noqa: F811
    monkeypatch.setattr(cells, "STRIPES", TALL)
    cells.test_cells_seeded_faceids_and_crop(renderer, stripe)


def test_queued_pairs_do_not_depend_on_the_order(renderer, stripe, capfd, monkeypatch):  # noqa: F811
    from esctp1raytracer_b200 import RNG_HASH, Camera

    name, s, W, H, eye, look = _cases()[0]
    cam = Camera.for_frame(eye, look, W, H)
    rs = renderer.upload(s)
    monkeypatch.setenv("TRACER_SHADOW_DIAG", "1")
    queued, frames = {}, {}
    for L in ("1", "4096", None):
        stripe(L)
        capfd.readouterr()
        a = renderer.trace(rs, cam, W, H, rng_mode=RNG_HASH, seed=5)
        _no_misses(a)
        q = [int(x) for x in re.findall(r"queued pairs (\d+)", capfd.readouterr().err)]
        assert q, "no shadow diagnostics line"
        queued[L], frames[L] = sum(q), a.rgb8
    assert queued["1"] > 1000, queued
    for L in ("4096", None):
        assert abs(queued[L] - queued["1"]) <= 0.03 * queued["1"], (L, queued)
        assert (frames[L] == frames["1"]).all(), L
