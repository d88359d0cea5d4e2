"""CPU checks of the seeded mode's row-count exchange between the calls that render one frame's bands (no GPU needed):

* the multi-GPU call's exchange between its per-GPU threads (tracer__row_exchange_host, the same RowExchange barrier and
  hook the call installs): every thread gets the frame's counts; a thread whose render failed before the exchange still
  arrives, so no thread waits, and every exchange then fails;
* dist.row_hits_all_reduce, the hook dist.render_frame passes, over a gloo process group of 2 and 3 ranks: every rank gets
  the frame's counts, zero-row ranks included.
"""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

from esctp1raytracer_b200 import _lib
from esctp1raytracer_b200.dist import band_rows_of_rank

I32P, U8P = C.POINTER(C.c_int32), C.POINTER(C.c_uint8)


def _own_rows(frame_rows, band_rows, world):
    """what each band's call offers: its own rows' counts, 0 elsewhere -> [world, H]"""
    H = len(frame_rows)
    out = np.zeros((world, H), np.int32)
    for r in range(world):
        rows = band_rows_of_rank(H, band_rows, r, world)
        out[r, rows] = frame_rows[rows]
    return out


def _exchange_threads(rows_in, fails):
    lib = _lib.load()
    lib.tracer__row_exchange_host.argtypes = [C.c_int32, C.c_int32, I32P, U8P, I32P, I32P]
    lib.tracer__row_exchange_host.restype = None
    n, H = rows_in.shape
    rows_in = np.ascontiguousarray(rows_in, np.int32)
    fails = np.ascontiguousarray(fails, np.uint8)
    out = np.full((n, H), -9, np.int32)
    rc = np.full(n, -9, np.int32)
    lib.tracer__row_exchange_host(n, H, rows_in.ctypes.data_as(I32P), fails.ctypes.data_as(U8P), out.ctypes.data_as(I32P),
                                  rc.ctypes.data_as(I32P))
    return out, rc


@pytest.mark.parametrize("n,H,B", [(2, 77, 8), (3, 50, 4), (8, 21, 8), (5, 9, 2)])
def test_multi_gpu_thread_exchange(n, H, B):
    rng = np.random.default_rng(n * 100 + H)
    frame_rows = rng.integers(0, 40, H).astype(np.int32)
    offered = _own_rows(frame_rows, B, n)
    out, rc = _exchange_threads(offered, np.zeros(n))
    assert (rc == 0).all() and (out == frame_rows).all()
    for failed in ([0], [n - 1], list(range(n))):  # GPUs whose render failed before the exchange
        fails = np.zeros(n)
        fails[failed] = 1
        out, rc = _exchange_threads(offered, fails)
        assert (rc[fails == 1] == -1).all() and (rc[fails == 0] != 0).all()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank(rank, world, port, frame_rows, B, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch.distributed as dist

    from esctp1raytracer_b200.dist import row_hits_all_reduce

    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        row_hits = _own_rows(frame_rows, B, world)[rank].copy()
        row_hits_all_reduce()(row_hits)
        q.put((rank, row_hits.tolist()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,H,B", [(2, 77, 8), (3, 10, 8)])  # (3, 10, 8): rank 2 renders no row
def test_dist_all_reduce_hook(world, H, B):
    frame_rows = np.random.default_rng(H).integers(0, 30, H).astype(np.int32)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, world, port, frame_rows, B, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert all(got[r] == frame_rows.tolist() for r in range(world))
