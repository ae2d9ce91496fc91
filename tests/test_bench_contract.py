"""bench.py --impl reference (the CPU arm the driver runs beside the GPU arm): one JSON line with the contract's
keys, runnable without a GPU. Uses the small C1 config so it takes seconds. Also --dump-outputs (what the timed
path computed, for comparing two builds) on both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from helpers import assert_close_fp32, fp32_tol


def test_reference_arm_json_line(tmp_path):
    env = dict(os.environ, PGCN_CACHE=str(tmp_path))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "C1",
                          "--steps", "3", "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    r = json.loads(lines[0])
    assert r["impl"] == "reference" and r["unit"] == "edges/s" and r["higher_is_better"] is True
    assert r["metric"].startswith("aggregated edges/sec") and r["steps"] == 3 and r["warmup"] == 1
    assert r["value"] > 0 and abs(r["value"] - (10556 + 2708) / (r["ms_per_step"] * 1e-3)) / r["value"] < 1e-6
    assert r["cpu_baseline"]["kind"] == "port" and r["cpu_baseline"]["cores"] >= 1 and r["cpu_baseline"]["value"] == r["value"]
    assert r["e2e"] == {"value": r["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert r["vs_baseline"] is None and r["dtype"] == "f32" and r["data"] == "synthetic" and "workload" in r["config"]


def test_reference_arm_other_ranks_exit_quietly(tmp_path):
    env = dict(os.environ, PGCN_CACHE=str(tmp_path), RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "C1",
                          "--gpus", "2", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "C1",
                          "--steps", "0"], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, PGCN_CACHE=str(tmp_path)))
    assert out.returncode != 0 and "--steps" in out.stderr and out.stdout.strip() == ""


def test_dump_rows_sample_is_fixed_and_within_budget():
    import bench
    from pgcn_b200 import graphio
    for config in ("C2", "C4", "C5"):
        n, _, f, _, _ = graphio.CONFIGS[config]
        for world in (1, 2, 8):
            m = n // world
            rows = bench.dump_rows(m, f, world)
            assert np.array_equal(rows, bench.dump_rows(m, f, world))
            assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < m
            assert world * rows.shape[0] * (4 * f + 8) <= bench.DUMP_BYTES < 64 * 10 ** 6
    assert np.array_equal(bench.dump_rows(2708, 16, 1), np.arange(2708))


def _c1_truth(H):
    from oracle import pgcn_oracle as orc
    from pgcn_b200 import graphio
    A = graphio.config_graph("C1")
    return orc.truth_forward(A, H), fp32_tol(A, H, int(orc.row_degree(A).max()))


def test_dump_outputs_reference_arm(tmp_path):
    """Every row of C1's aggregation (it fits), the same bits on a second run, equal to the fp64 truth of the
    seeded input within the fp32 bound."""
    env = dict(os.environ, PGCN_CACHE=str(tmp_path / "cache"))
    dumps = []
    for i in range(2):
        d = tmp_path / ("dump%d" % i)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "C1",
                              "--steps", "2", "--warmup", "1", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, env=env)
        assert out.returncode == 0, out.stderr[-2000:]
        assert sorted(os.listdir(d)) == ["Z.npy", "Z_rows.npy"]
        dumps.append((np.load(d / "Z.npy"), np.load(d / "Z_rows.npy")))
    Z, rows = dumps[0]
    assert Z.dtype == np.float32 and Z.shape == (2708, 16) and rows.dtype == np.float64
    assert np.array_equal(rows, np.arange(2708)) and np.array_equal(Z, dumps[1][0])
    H = np.random.RandomState(1).uniform(-1, 1, size=(2708, 16)).astype(np.float32)     # bench.run_reference's input
    Z64, tol = _c1_truth(H)
    assert_close_fp32(Z, Z64, tol, "reference arm dump")


@pytest.mark.gpu
def test_dump_outputs_gpu_arm(tmp_path):
    """The GPU arm's dump is the Z of its last timed step: the seeded input regenerated here, aggregated in fp64,
    matches within the fp32 bound; exactly --steps steps were timed."""
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: -m gpu tests must run on the B200 box")
    d = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "C1", "--steps", "7",
                          "--warmup", "3", "--no-cpu-baseline", "--no-lib-baseline", "--no-e2e", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600, env=dict(os.environ, PGCN_CACHE=str(tmp_path / "cache")))
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads(out.stdout.strip())
    assert r["steps"] == 7 and r["gpu_launches"] > 0 and r["gpu_launches"] % 7 == 0
    Z, rows = np.load(d / "Z.npy"), np.load(d / "Z_rows.npy")
    assert Z.dtype == np.float32 and Z.shape == (2708, 16) and np.array_equal(rows, np.arange(2708))
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1)                                  # bench.main's input, rank 0
    H = ((torch.rand((2708, 16), device=dev, generator=gen) * 2 - 1)).cpu().numpy()
    Z64, tol = _c1_truth(H)
    assert_close_fp32(Z, Z64, tol, "GPU arm dump")
