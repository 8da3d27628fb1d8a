"""bench.py's contract: the reference arm prints one JSON line with the agreed keys, --dump-outputs writes a bounded
sample that is the same from run to run and (GPU) equals what the headline solve returns, and the product arm refuses
to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=300):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_prints_one_json_line(oracle_built):
    proc = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample", "4", "--batch", "64"])
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout carries the one JSON line only"
    line = json.loads(lines[0])
    assert line["impl"] == "reference"
    assert line["metric"] == "optimized_trajectories_per_sec" and line["unit"] == "trajectories/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 2
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["config"]["config"] == "C4" and "workload" in line["config"]          # the north star's headline config
    assert len(line["cpu_baseline"]["step_seconds"]) == 2
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    # the CPU arm never maps the product's CUDA library (its solves run on oracle/ only)
    probe = subprocess.run([sys.executable, "-c",
                            "import sys; sys.path.insert(0, %r); import bench; b = bench.make_batch('C4', 16); "
                            "from trajectory_generator_b200 import synthetic; synthetic.container_for(b.take([1, 2]), 0); "
                            "print(any('libTrajectoryConstraints' in l and 'oracle' not in l for l in open('/proc/self/maps')))" % ROOT],
                           capture_output=True, text=True, cwd=ROOT)
    assert probe.stdout.strip() == "False", probe.stdout + probe.stderr
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == line["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_dump_outputs_is_a_bounded_reproducible_sample(tmp_path):
    import numpy as np
    import torch
    import bench
    B, n = 262144, 34                                   # the headline batch: its outputs exceed the 64 MB cap
    out = {"x": torch.arange(B * n, dtype=torch.float64).reshape(B, n), "f": torch.arange(B, dtype=torch.float64),
           "status": torch.arange(B, dtype=torch.int32) % 10, "nit": torch.arange(B, dtype=torch.int32)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), out)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["f.npy", "nit.npy", "status.npy", "x.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    arr = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    rows = arr["nit"].astype(np.int64)
    assert all(a.dtype == np.float64 and len(a) == len(rows) for a in arr.values()) and 0 < len(rows) < B
    assert np.all(np.diff(rows) > 0)
    assert np.array_equal(arr["x"], out["x"].numpy()[rows]) and np.array_equal(arr["status"], rows % 10)
    assert all(np.array_equal(arr[f[:-4]], np.load(tmp_path / "b" / f)) for f in files)


@pytest.mark.gpu
def test_dump_outputs_are_what_the_headline_solve_returns(native_lib, tmp_path):
    """bench.py --dump-outputs on a small headline batch: the files equal a direct batch.solve of the same seeded batch"""
    import numpy as np
    import torch
    import bench
    from trajectory_generator_b200 import batch as tgb
    proc = _run(["--quick", "--no-cpu-baseline", "--batch", "512", "--steps", "2", "--warmup", "1",
                 "--dump-outputs", str(tmp_path)], timeout=600)
    assert proc.returncode == 0, proc.stderr[-2000:]
    bt = bench.make_batch("C4", 512)
    dev = torch.device("cuda:0")
    out = tgb.solve(bt.spec, torch.from_numpy(bt.par).to(dev), torch.from_numpy(bt.x0).to(dev), jacobian="fd")
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in out)
    for k, v in out.items():
        assert np.array_equal(np.load(tmp_path / (k + ".npy")), v.cpu().numpy().astype(np.float64)), k


def test_product_arm_needs_a_cuda_device(native_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    proc = _run(["--steps", "1", "--warmup", "0", "--no-cpu-baseline"], env={"TG_BENCH_CUDA_RETRY": "4"}, timeout=120)
    assert proc.returncode != 0
    assert "no CUDA device" in (proc.stderr + proc.stdout)
    assert not [ln for ln in proc.stdout.splitlines() if ln.strip().startswith("{")], "no number without a device"
