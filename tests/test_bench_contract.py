"""Tests of the bench.py contract: the reference arm prints ONE JSON line with the agreed keys
(metric / unit / value / impl / cpu_baseline / e2e ...) and times the reference's own kernel; --dump-outputs
writes what the timed path computed (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import scaled_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--workload", "cfg1"], capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "NLMeansFilter Mvoxel/s" and d["unit"] == "Mvoxel/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"] == "cfg1" and d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1"],
                       capture_output=True, text=True, timeout=60, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_sample_is_fixed_and_bounded():
    import bench
    y, x, t = bench.dump_sample((4096, 4096, 32, 4), 1)
    assert len(y) * 4 * 4 <= 64 << 20 and len(y) > 1 << 20
    flat = (y * 4096 + x) * 32 + t
    assert (np.diff(flat) > 0).all() and flat[-1] < 4096 * 4096 * 32
    assert all(np.array_equal(a, b) for a, b in zip((y, x, t), bench.dump_sample((4096, 4096, 32, 4), 1)))
    assert 4 * len(bench.dump_sample((16384, 16384, 64, 4), 4)[0]) * 4 * 4 <= 64 << 20
    y, x, t = bench.dump_sample((3, 5, 2, 4), 1)                        # small results are written whole
    assert np.array_equal((y * 5 + x) * 2 + t, np.arange(30))


def _bench_dump(tmp_path, *args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-e2e", "--no-cpu",
                        "--dump-outputs", str(tmp_path)] + list(args), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout)["steps"] == int(args[args.index("--steps") + 1])
    assert os.listdir(tmp_path) == ["out.npy"]
    return np.load(tmp_path / "out.npy")


@pytest.mark.gpu
def test_dump_outputs_of_the_real_raster_are_the_reference_output(tmp_path):
    got = _bench_dump(tmp_path, "--workload", "cfg1", "--steps", "2", "--warmup", "1")
    want = np.load(os.path.join(ROOT, "tests", "golden", "slc_cfg1.npz"))["out_as_written"].reshape(-1, 4)
    assert got.dtype == np.float32 and got.shape == want.shape
    assert scaled_err(got, want) < 1e-4


@pytest.mark.gpu
def test_dump_outputs_of_a_streamed_workload_sample_the_last_step(tmp_path):
    import torch
    import bench
    from nd_b200 import device
    got = _bench_dump(tmp_path, "--workload", "cfg4", "--global-rows", "24", "--steps", "2", "--warmup", "1")
    wl = bench.WORKLOADS["cfg4"]
    shape = (24, wl["nx"], wl["nt"], wl["V"])
    whole = device.Plan(shape, wl["r"], bench.fvec(wl), wl["sigma"], wl["h"]).apply(
        device.synth_cube(*shape, seed=42))
    y, x, t = (torch.from_numpy(a).cuda() for a in bench.dump_sample(shape, 1))
    want = whole[y, x, t].cpu().numpy()
    assert got.dtype == np.float32 and got.shape == want.shape and len(got) < 24 * wl["nx"] * wl["nt"]
    assert scaled_err(got, want) < 1e-4
