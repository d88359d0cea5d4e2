"""Row-band sharding of one frame across the GPUs of a box (one process per GPU).

The reference has no multi-device path; its closest analogue is thread-per-row
(src/main.cpp:629-643).  Pixels are independent, so the frame's PPM rows are cut
into bands of ``band_rows`` rows and band b goes to rank ``b % world``
(interleaved, to balance coverage-dependent shadow cost).  The scene is replicated.
The ONE exchange step is the gather of the packed 8-bit bands to rank 0
(torch.distributed -> NCCL over NVLink); rank 0 then scatters the band-packed
buffers into PPM order with ``tracer_cuda_assemble_bands``.

The counter-based RNG is keyed by the image index, so the assembled frame is
byte-identical to a single-GPU frame (tests/test_gpu_parity.py, tests/test_dist_gloo.py).
The seeded std::mt19937 mode needs one more exchange per frame: each rank's per-row hit
counts, all-reduced (SUM) over the group, give every rank its hits' places in the stream.
"""
from __future__ import annotations

import numpy as np

DEFAULT_BAND_ROWS = 8


def band_rows_of_rank(height: int, band_rows: int, rank: int, world: int) -> np.ndarray:
    """PPM rows (row 0 = h=H-1) rendered by ``rank``, in the order they are packed."""
    pr = np.arange(height)
    return pr[(pr // band_rows) % world == rank]


def padded_rows(height: int, band_rows: int, world: int) -> int:
    """rows in every rank's gather buffer (the largest share, so all buffers are equal)"""
    return max(len(band_rows_of_rank(height, band_rows, r, world)) for r in range(world))


def gather_bands(local, rank: int, world: int, dst: int = 0, group=None):
    """Gather equal-sized band buffers (torch tensors, CUDA for NCCL / CPU for gloo) to ``dst``.
    Returns the stacked [world, ...] tensor on ``dst``, None elsewhere."""
    import torch
    import torch.distributed as dist

    if world == 1:
        return local.unsqueeze(0)
    out = None
    if rank == dst:
        stacked = torch.empty((world,) + tuple(local.shape), dtype=local.dtype, device=local.device)
        out = list(stacked.unbind(0))
    dist.gather(local, out, dst=dst, group=group)
    return stacked if rank == dst else None


def torch_stream_handle():
    """cudaStream_t of torch's current stream, as the C ABI wants it.  torch reports the legacy default stream as
    handle 0, which the ABI reads as "use the library's own (non-blocking) stream": the render would then not be
    ordered with torch's allocations, the NCCL gather and the assemble kernel.  cudaStreamLegacy (0x1) names the
    same stream explicitly."""
    import torch

    return torch.cuda.current_stream().cuda_stream or 1


def row_hits_all_reduce(group=None):
    """The seeded mode's exchange hook for ``Renderer.trace(row_hits_exchange=...)``: every rank's per-row hit counts
    summed over the process group, in place (each row has one owner, so the sum is the frame's counts)."""

    def exchange(row_hits):
        import torch
        import torch.distributed as dist

        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        t = torch.from_numpy(row_hits.copy()).to(dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        row_hits[:] = t.cpu().numpy()

    return exchange


def render_frame(renderer, resident_scene, camera, width, height, *, rank=0, world=1, band_rows=DEFAULT_BAND_ROWS,
                 rng_mode=0, seed=1, group=None, bundle_cull=False, samples_per_pixel=0, bvh=False):
    """Render this rank's bands into HBM, gather to rank 0, assemble.  Returns
    (frame uint8 CUDA tensor [H, W, 3] on rank 0 else None, per-rank stats dict).  To move geometry between frames,
    every rank calls ``resident_scene.update(...)`` on its own scene with the same arrays before this call."""
    import torch

    rows_pad = padded_rows(height, band_rows, world) if world > 1 else height
    local = torch.zeros((rows_pad, width, 3), dtype=torch.uint8, device="cuda")
    stream = torch_stream_handle()
    bands = (band_rows, rank, world) if world > 1 else None
    exchange = row_hits_all_reduce(group) if world > 1 and rng_mode == 1 else None  # RNG_MT19937
    fr = renderer.trace(resident_scene, camera, width, height, rng_mode=rng_mode, seed=seed, bands=bands,
                        out_device_ptr=local.data_ptr(), stream=stream, bundle_cull=bundle_cull, bvh=bvh,
                        samples_per_pixel=samples_per_pixel, row_hits_exchange=exchange)
    if world == 1:
        return local, fr.stats
    gathered = gather_bands(local, rank, world, 0, group)
    frame = None
    if rank == 0:
        frame = torch.empty((height, width, 3), dtype=torch.uint8, device="cuda")
        renderer.assemble_bands(gathered.data_ptr(), frame.data_ptr(), width, height, band_rows, world, rows_pad,
                                stream=stream)
    return frame, fr.stats
