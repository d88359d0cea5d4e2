"""bench.py's own arm, dry-run on the CPU: the GPU-facing calls (Renderer, dist.render_frame, torch.cuda events / pinned
memory) are replaced by stand-ins that return plausible frame statistics, everything else — argument handling, the timed
loop, the roofline arithmetic, the JSON line — is bench.py's real code.  Asserts that the line carries every key the
measurement contract names and that the derived numbers follow from the statistics.  (The numbers themselves are only
meaningful on the B200: tests/test_gpu_*.py and the committed profiles/ hold those.)
"""
import io
import json
import os
import subprocess
import sys
from contextlib import redirect_stdout

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_standins import MS_PRIMARY, MS_SHADOW, PAIRS_PRIMARY, PAIRS_SHADOW, PAIRS_SHADOW_REF, install


@pytest.fixture
def dry_bench(monkeypatch):
    import bench

    install(monkeypatch.setattr)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)

    def run(*argv):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        buf = io.StringIO()
        with redirect_stdout(buf):
            bench.main()
        lines = [l for l in buf.getvalue().splitlines() if l.startswith("{")]
        assert len(lines) == 1, buf.getvalue()
        return json.loads(lines[0])

    return run


def test_bench_line_has_the_contract_keys_and_consistent_arithmetic(dry_bench):
    d = dry_bench("--workload", "small", "--tris", "3000", "--width", "64", "--height", "48", "--steps", "4", "--warmup", "3",
                  "--no-cpu-baseline")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "frame_sha256"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] == 3 and d["higher_is_better"] is True
    assert d["dtype"] == "f32" and d["vs_baseline"] is None and d["scaling"] == "strong" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"] and d["config"]["mode"] == "brute"
    assert "l2_policy" in d["config"]
    assert d["gpu_launches"] == 21 * 4
    rays = 64 * 48 + 64 * 48 // 2 * 4
    assert d["rays_per_step"] == rays
    assert d["value"] == pytest.approx(rays / (d["ms_per_step"] * 1e-3) / 1e6)
    e = d["e2e"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in e, k
    assert e["d2h_bytes_per_step"] == 64 * 48 * 3 and e["h2d_bytes_per_step"] > 3000 * 36
    assert "tracer_cuda_render" in e["path"]
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["peak"] == 68.0 and r["unit"] == "TFLOP/s"
    sweep_s = (MS_PRIMARY + MS_SHADOW) * 1e-3
    want = (4.25 * PAIRS_PRIMARY + 5.0 * PAIRS_SHADOW_REF) / sweep_s / 1e12  # algorithmic pairs, per launch-time of both sweeps
    assert r["achieved"] == pytest.approx(want) and r["frac"] == pytest.approx(want / 68.0)
    assert r["primary_tflops"] == pytest.approx(4.25 * PAIRS_PRIMARY / (MS_PRIMARY * 1e-3) / 1e12)
    assert r["shadow_tflops"] == pytest.approx(5.0 * PAIRS_SHADOW / (MS_SHADOW * 1e-3) / 1e12)  # swept pairs here
    dk = r["dominant_kernel"]
    assert dk["kernel"].startswith("trk::primary_kernel")
    assert dk["achieved"] == pytest.approx(r["primary_tflops"]) and dk["frac"] == pytest.approx(r["primary_tflops"] / 68.0)
    assert dk["share_of_sweep_time"] == pytest.approx(MS_PRIMARY / (MS_PRIMARY + MS_SHADOW))
    assert r["as_issued"]["flop_per_pair"] == {"primary": 6.25, "shadow": 7.0}
    assert r["fma_pipe"]["lane_ops_per_pair"] == {"primary": 3.125, "shadow": 3.5}
    assert r["mix_ceiling_frac"] == pytest.approx((4.25 * PAIRS_PRIMARY + 5.0 * PAIRS_SHADOW_REF) /
                                                  (2 * (3.125 * PAIRS_PRIMARY + 3.5 * PAIRS_SHADOW_REF)))
    assert d["clocks"]["reasons"] in (["nvidia-smi unavailable"], []) or isinstance(d["clocks"]["reasons"], list)
    oc = d["optional_bundle_cull_mode"]
    assert oc["frame_identical_to_default_mode"] is True


def test_bench_refuses_to_run_without_a_gpu(monkeypatch):
    import torch

    import bench

    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # also on a machine that has one
    monkeypatch.setattr(sys, "argv", ["bench.py", "--no-cpu-baseline"])
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    with pytest.raises(SystemExit) as ei:
        bench.main()
    assert "no CPU fallback" in str(ei.value)


@pytest.mark.parametrize("argv", [
    ("--workload", "c1", "--steps", "3", "--warmup", "3", "--no-cpu-baseline"),
    ("--workload", "c3", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--no-cull"),
    ("--workload", "small", "--tris", "2000", "--width", "32", "--height", "24", "--mode", "cull", "--no-cpu-baseline"),
    ("--workload", "c5", "--tris", "2000", "--width", "32", "--height", "24", "--no-cpu-baseline", "--no-cull"),
])
def test_bench_flag_combinations_produce_one_line(dry_bench, argv):
    d = dry_bench(*argv)
    assert d["metric"].startswith("Mrays/s") and d["value"] > 0 and d["roofline"]["frac"] > 0
    if "--no-e2e" in argv:
        assert d["e2e"] is None
    if "c5" in argv:
        assert d["config"]["spp"] == 16


@pytest.mark.parametrize("size,sampled", [((64, 48), False), ((3840, 2160), True)])
def test_bench_dump_outputs_writes_the_last_timed_frame(dry_bench, monkeypatch, tmp_path, size, sampled):
    """--steps sets the number of timed renders; --dump-outputs writes the last one's frame as float32 (a fixed pixel sample
    when the whole frame would exceed 64 MB), the same files on every run"""
    import numpy as np
    import torch

    from esctp1raytracer_b200 import dist as tdist

    fake = tdist.render_frame
    calls = []

    def render_frame(renderer, rs, cam, W, H, **kw):
        frame, st = fake(renderer, rs, cam, W, H, **kw)
        calls.append(1)
        frame = torch.from_numpy(np.random.default_rng(len(calls)).integers(0, 256, (H, W, 3), dtype=np.uint8))
        return frame, st

    monkeypatch.setattr(tdist, "render_frame", render_frame)
    W, H = size
    dumps = []
    for run in range(2):
        calls.clear()
        out = tmp_path / f"run{run}"
        dry_bench("--workload", "small", "--tris", "2000", "--width", str(W), "--height", str(H), "--steps", "5", "--warmup", "2",
                  "--no-cpu-baseline", "--no-e2e", "--no-cull", "--dump-outputs", str(out))
        assert len(calls) == 2 + 5
        files = sorted(p.name for p in out.iterdir())
        dumps.append({f: np.load(out / f) for f in files})
    last = np.random.default_rng(7).integers(0, 256, (H, W, 3), dtype=np.uint8)  # the frame of the 7th call
    a, b = dumps
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20 and all(v.dtype in (np.float32, np.float64) for v in a.values())
    if sampled:
        assert sorted(a) == ["frame_sample.npy", "frame_sample_pixel.npy"]
        idx = a["frame_sample_pixel.npy"].astype(np.int64)
        assert len(np.unique(idx)) == len(idx) and np.array_equal(a["frame_sample.npy"], last.reshape(-1, 3)[idx].astype(np.float32))
    else:
        assert sorted(a) == ["frame.npy"] and np.array_equal(a["frame.npy"], last.astype(np.float32))


def test_bench_refuses_dump_outputs_with_the_reference_arm(monkeypatch, tmp_path, capsys):
    import bench

    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--dump-outputs", str(tmp_path / "d")])
    with pytest.raises(SystemExit) as ei:
        bench.main()
    assert ei.value.code == 2 and "--dump-outputs" in capsys.readouterr().err and not (tmp_path / "d").exists()


def test_bench_torchrun_path_two_ranks_on_gloo():
    """the path the driver's scaling runs take (torchrun, one rank per GPU): reductions over ranks, rank 0 prints ONE line"""
    port = 29600 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "bench_dryrun_worker.py"), "--gpus", "2", "--steps", "3", "--warmup", "3",
           "--workload", "small", "--tris", "2000", "--width", "64", "--height", "48", "--no-cpu-baseline"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and d["steps"] == 3 and "torchrun" in d["multi_gpu_path"]
    assert d["rays_per_step"] == 64 * 48 + 64 * 48 // 2 * 4          # the two half-frame shares add up to the frame
    assert d["gpu_launches"] == (21 * 3) * 2 + 3                       # both ranks' kernels + rank 0's assemble per step
    r_ = d["roofline"]
    # per-GPU rate: each rank sweeps half of the pairs in half of the time
    assert r_["achieved"] == pytest.approx((4.25 * PAIRS_PRIMARY + 5.0 * PAIRS_SHADOW_REF) / ((MS_PRIMARY + MS_SHADOW) * 1e-3) / 1e12, rel=1e-3)
    assert r_["dominant_kernel"]["frac"] == pytest.approx(4.25 * PAIRS_PRIMARY / (MS_PRIMARY * 1e-3) / 1e12 / 68.0, rel=1e-3)
    assert d["e2e"]["h2d_bytes_per_step"] > 2 * 2000 * 36 and "per rank" in d["e2e"]["path"]
    assert d["frame_sha256"] and d["optional_bundle_cull_mode"]["frame_identical_to_default_mode"] is True
