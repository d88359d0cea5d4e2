"""CPU checks of the device replay of the seeded draws (csrc/mt19937.cuh) through the library's host build of the same
source (tracer__mt19937_words_host, tracer__mt19937_replay_host, tracer__mt19937_band_ordinals_host: no GPU needed).

* the stream, generated in 227-word steps, equals std::mt19937 compiled by g++: positions 0-2000, around multiples of 624
  and near 10^7;
* the chunked automaton's faceIDs equal tracer_mt19937_faceids (the sequential replay) on the golden frames' hit masks, on
  random masks with 0-4 lights and face counts that never / often reject (3 * 2^29 and 1.5e9 reject 25-30 % of draws,
  so the first stream is short and runs of rejections cross chunk boundaries), for chunks of 1, 2, 3L-1, 3L and 4096 words;
* the hit ordinals of a band selection (own row counts, the exchanged ones, the scan over rows, the in-row rank) equal
  a cumulative sum over the whole frame's mask in scan order.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from conftest import golden_names, load_golden

from esctp1raytracer_b200 import _lib
from esctp1raytracer_b200.dist import band_rows_of_rank

U8P, I32P, I64P, U32P = (C.POINTER(t) for t in (C.c_uint8, C.c_int32, C.c_int64, C.c_uint32))


def _p(a, t):
    return a.ctypes.data_as(t)


@pytest.fixture(scope="module")
def lib():
    lib = _lib.load()
    lib.tracer__mt19937_words_host.argtypes = [C.c_uint32, C.c_int64, C.c_int64, U32P]
    lib.tracer__mt19937_words_host.restype = None
    lib.tracer__mt19937_replay_host.argtypes = [C.c_uint32, C.c_int32, I32P, C.c_int64, U8P, C.c_int64, I32P]
    lib.tracer__mt19937_replay_host.restype = C.c_int64
    lib.tracer__mt19937_band_ordinals_host.argtypes = [C.c_int32] * 5 + [U8P, I64P]
    lib.tracer__mt19937_band_ordinals_host.restype = C.c_int
    return lib


def reference_faceids(lib, faces, W, H, seed, hit_img):
    """tracer_mt19937_faceids over a scene whose light l is a geometry of faces[l] triangles: [H*W, L], image order"""
    L = len(faces)
    off = np.zeros(2 * max(L, 1), np.int32)  # geometry 2l spans [0, F_l): no offset sum can overflow int32
    off[1::2][:L] = faces
    lg = np.arange(0, 2 * L, 2, dtype=np.int32)
    cs = _lib.SceneFlat()
    cs.n_geoms, cs.geom_tri_offset, cs.n_lights, cs.light_geom = 2 * max(L, 1) - 1, _p(off, I32P), L, _p(lg, I32P)
    hit = np.ascontiguousarray(hit_img, np.uint8).reshape(-1)
    out = np.full((W * H, L), -7, np.int32)
    _lib.check(lib.tracer_mt19937_faceids(C.byref(cs), W, H, seed, _p(hit, U8P), _p(out, I32P)))
    return out


def replay(lib, faces, W, H, seed, hit_img, chunk):
    """the host build of the device replay, on the scan-order mask; -> ([H*W, L] image order, stream words used)"""
    L = len(faces)
    hit_scan = np.ascontiguousarray(np.asarray(hit_img, np.uint8).reshape(H, W)[::-1]).reshape(-1)
    f = np.asarray(faces, np.int32)
    out = np.full((W * H, L), -7, np.int32)
    D = lib.tracer__mt19937_replay_host(seed, L, _p(f, I32P), W * H, _p(hit_scan, U8P), chunk, _p(out, I32P))
    return out.reshape(H, W, L)[::-1].reshape(W * H, L), D


def chunks(L):
    return sorted({1, 2, 4096} | ({3 * L - 1, 3 * L} if L else set()))


def test_stream_equals_std_mt19937(lib, tmp_path):
    src = tmp_path / "mt.cpp"
    src.write_text("#include <random>\n#include <cstdio>\n#include <cstdlib>\n#include <cstdint>\n"
                   "int main(int c, char **v){ std::mt19937 g((uint32_t)std::strtoul(v[1],0,10)); long n = std::atol(v[2]);"
                   " for (long i = 0; i < n; ++i) { uint32_t y = g(); std::fwrite(&y, 4, 1, stdout); } return 0; }\n")
    exe = tmp_path / "mt"
    subprocess.check_call(["g++", "-std=c++17", "-O2", str(src), "-o", str(exe)])
    for seed in (5489, 1, 0xDEADBEEF):
        n = 10_000_010
        want = np.frombuffer(subprocess.run([str(exe), str(seed), str(n)], capture_output=True, check=True).stdout, np.uint32)
        spots = [(0, 2001), (10_000_000 - 700, 710)] + [(max(0, 624 * k - 5), 11) for k in (1, 2, 3, 10, 227, 1000)]
        for start, cnt in spots:
            got = np.zeros(cnt, np.uint32)
            lib.tracer__mt19937_words_host(seed, start, cnt, _p(got, U32P))
            assert np.array_equal(got, want[start:start + cnt]), (seed, start)


@pytest.mark.parametrize("name", golden_names())
def test_automaton_equals_sequential_replay_on_golden_frames(lib, name):
    fs, fr = load_golden(name)
    W, H, seed = fr["W"], fr["H"], fr["seed"]
    faces = (fs.geom_tri_offset[fs.light_geom + 1] - fs.geom_tri_offset[fs.light_geom]).astype(np.int32)
    hit = fr["tri"] >= 0
    want = reference_faceids(lib, faces, W, H, seed, hit)
    assert np.array_equal(want, fr["faceid"])
    for chunk in chunks(len(faces)):
        got, _ = replay(lib, faces, W, H, seed, hit, chunk)
        assert np.array_equal(got, want), chunk


FACES = [1, 2, 3, 10, 100, 173, 250, 2 ** 31 - 1, 3 * 2 ** 29, 1_500_000_000]
REJECTING = (3 * 2 ** 29, 1_500_000_000)  # 2^32 mod F = 2^30 and 1.29e9: 25 % and 30 % of draws rejected


@pytest.mark.parametrize("L", [0, 1, 2, 3, 4])
def test_automaton_equals_sequential_replay_on_random_masks(lib, L):
    rng = np.random.default_rng(100 + L)
    W, H = 37, 23
    for trial in range(4):
        faces = list(rng.choice(FACES, size=L)) if trial else [REJECTING[i % 2] for i in range(L)]
        hit = rng.random(W * H) < rng.choice([0.05, 0.6, 1.0])
        seed = int(rng.integers(0, 2 ** 32))
        want = reference_faceids(lib, faces, W, H, seed, hit)
        for chunk in chunks(L):
            got, D = replay(lib, faces, W, H, seed, hit, chunk)
            assert np.array_equal(got, want), (faces, chunk)
        if trial == 0 and L and hit.sum() > 10:  # rejections left the first stream (3 L T words) short
            assert D > 3 * L * hit.sum()


def test_rejection_runs_cross_chunk_boundaries(lib):
    """with chunks of 3L-1 and 3L words, a chunk boundary falls inside a run of two or more rejected draws"""
    faces, W, H, seed = [3 * 2 ** 29, 1_500_000_000], 64, 40, 77
    hit = np.ones(W * H, bool)
    want = reference_faceids(lib, faces, W, H, seed, hit)
    y = np.zeros(3 * 2 * W * H * 2, np.uint32)
    lib.tracer__mt19937_words_host(seed, 0, len(y), _p(y, U32P))
    for chunk in (5, 6, 4096):
        assert np.array_equal(replay(lib, faces, W, H, seed, hit, chunk)[0], want)
    # the sequential consumption, to find the runs: (position, light) of every rejected faceID draw
    F = np.array(faces, np.uint64)
    thr = (2 ** 32) % F
    i, rejected = 0, []
    for _ in range(W * H):
        for l in range(2):
            while True:
                low = (int(y[i]) * int(F[l])) & 0xFFFFFFFF
                i += 1
                if low < F[l] and low < thr[l]:
                    rejected.append(i - 1)
                    continue
                break
            i += 2
    r = np.array(rejected)
    runs = r[1:][np.diff(r) == 1]  # second word of a run of rejections
    assert len(runs) and any(((runs % c) == 0).any() for c in (5, 6))


@pytest.mark.parametrize("band_rows,band_count", [(2, 8), (3, 5), (4, 8), (8, 16)])
def test_band_hit_ordinals(lib, band_rows, band_count):
    rng = np.random.default_rng(band_rows * 100 + band_count)
    W, H = 29, 37  # (8, 16): 5 bands, so band indices 5..15 render no row
    hit = rng.random(H * W) < 0.55
    hit[(H - 1 - 3) * W:(H - 1 - 3) * W + W] = False  # an empty row
    scan = hit.reshape(H, W)[::-1]  # PPM row order
    ordinal = np.where(scan, np.cumsum(scan.reshape(-1)).reshape(H, W) - 1, -1)
    empty = 0
    for bi in range(band_count):
        rows = band_rows_of_rank(H, band_rows, bi, band_count)
        out = np.full(max(len(rows), 1) * W, -9, np.int64)
        n = lib.tracer__mt19937_band_ordinals_host(W, H, band_rows, bi, band_count, _p(hit.astype(np.uint8), U8P), _p(out, I64P))
        assert n == len(rows)
        empty += n == 0
        assert np.array_equal(out[:n * W].reshape(n, W), ordinal[rows])
    assert (band_count * band_rows > H) == (empty > 0)
    # the whole frame is the same code with its own counts being the frame's
    out = np.zeros(H * W, np.int64)
    assert lib.tracer__mt19937_band_ordinals_host(W, H, 0, 0, 1, _p(hit.astype(np.uint8), U8P), _p(out, I64P)) == H
    assert np.array_equal(out.reshape(H, W), ordinal)
