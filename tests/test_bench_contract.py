"""bench.py contract checks that need no GPU: the reference arm (CPU oracle) prints one JSON line with the
required keys, and the GPU arm's JSON (checked on the GPU box) carries roofline / cpu_baseline / e2e."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert BASE_KEYS <= set(line)
    assert line["impl"] == "reference" and line["unit"] == "trajectories/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["dtype"] == "f64" and line["vs_baseline"] is None
    assert line["scaling"] == "strong" and line["config"]["total_trajectories"] == 1048576
    # both arms print the same config dict (the driver's same_config check)
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.config_dict("C5", 1048576)
    cb = line["cpu_baseline"]
    assert cb["cpu_info"]["effective"] >= cb["cores"] >= 1 and cb["per_core"] > 0


@pytest.mark.gpu
def test_gpu_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "3",
                          "--no-cpu-baseline", "--no-extras"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert BASE_KEYS <= set(line)
    assert line["results_ok"] and line["gpu_launches"] == 5
    r = line["roofline"]
    assert r["bound"] == "hbm" and 0.05 < r["frac"] < 1.2 and r["unit"] == "GB/s"
    assert abs(r["achieved"] / r["peak"] - r["frac"]) < 1e-9
    e = line["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert e["bitwise_equal_to_device_path"]
    assert line["clocks"]["sm_mhz"] is not None
    assert line["scaling"] == "strong" and line["config"]["total_trajectories"] == 1048576
    assert line["shard"]["trajectories_per_gpu"] == 1048576


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_path_outputs(tmp_path, solver):
    """--dump-outputs writes float64 .npy files (<= 64 MB in all) holding exactly the sampled rows of a fresh solve of
    the bench's seeded batch (the whole batch: kernel routing depends on the batch size), the same on a second run."""
    import numpy as np
    import torch
    import mav_trajectory_generation_b200 as m
    sys.path.insert(0, ROOT)
    import bench
    total = 65536
    dumps = []
    for run in range(2):
        d = tmp_path / str(run)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                              "--total", str(total), "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        files = sorted(p.name for p in d.iterdir())
        assert files == ["coeffs.npy", "rows.npy", "status.npy"]
        assert sum(p.stat().st_size for p in d.iterdir()) <= 64 << 20
        arrays = {f[:-4]: np.load(d / f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        dumps.append(arrays)
    for k in dumps[0]:
        assert np.array_equal(dumps[0][k], dumps[1][k]), k
    rows, coeffs, status = dumps[0]["rows"].astype(np.int64), dumps[0]["coeffs"], dumps[0]["status"]
    assert len(rows) > 1000 and (np.diff(rows) > 0).all() and (status == 0).all()
    N, r, K, D, _ = bench.CONFIGS["C5"]
    _, times, dfix = bench.synth_batch(torch, N, K, D, total, torch.device("cuda:0"), seed=1234)
    want = solver.solve_linear(m.Problem(N, r, K, D), times, dfix)
    assert np.array_equal(want[torch.from_numpy(rows).cuda()].cpu().numpy(), coeffs)
