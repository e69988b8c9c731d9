"""bench.py's reference arm runs without a GPU (it times the torch-CPU port of the path), so its JSON line -- the
contract the driver parses -- is checked here; the kdcc arm needs a B200 and must refuse to run without one."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, capture_output=True, text=True,
                          timeout=timeout)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--crop", "256"], 600)   # small crop: seconds, same line
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["unit"] == "img/s"
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["vs_baseline"] is None


def test_kdcc_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--e2e-steps", "0"], 300)
    assert r.returncode != 0
    assert "cuda" in (r.stderr + r.stdout).lower()


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample_of_large_ones(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 1000)
    big = torch.arange(5000, dtype=torch.float32).reshape(50, 100)
    arrays = {"small": torch.tensor([1.5, -2.0], dtype=torch.bfloat16), "scalar": torch.tensor(0.25, dtype=torch.float64), "big": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    small, scalar = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "scalar.npy")
    assert small.dtype == np.float32 and small.tolist() == [1.5, -2.0]
    assert scalar.dtype == np.float64 and scalar.shape == () and float(scalar) == 0.25
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (1000,) and np.array_equal(a, b)
    assert len(np.unique(a)) == 1000 and np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < 5000   # distinct, ordered, in range


def test_reference_arm_refuses_dump_outputs(tmp_path):
    r = _run(["--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path)], 300)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_kdcc_arm_dumps_its_last_timed_step(tmp_path):
    """Two runs with the same arguments: the dump holds the last timed step (its hint loss is the one the JSON line reports),
    stays under 64 MB of float arrays, and the runs agree (the inputs are seeded)."""
    import numpy as np
    args = ["--steps", "2", "--warmup", "1", "--batch", "1", "--no-cpu-baseline", "--no-gpu-baseline", "--no-extras", "--e2e-steps", "0"]
    dumps = []
    for d in ("a", "b"):
        r = _run(args + ["--dump-outputs", str(tmp_path / d)], 600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2
        files = sorted(os.listdir(tmp_path / d))
        assert {"hint_loss.npy", "kd_loss.npy", "params.npy", "grads.npy", "input_grad_site1.npy"} <= set(files), files
        assert sum(os.path.getsize(tmp_path / d / f) for f in files) <= 64 << 20
        dump = {f[:-4]: np.load(tmp_path / d / f) for f in files}
        assert all(v.dtype in (np.float32, np.float64) for v in dump.values())
        assert abs(float(dump["hint_loss"]) - line["losses"]["hint"]) <= 1e-6 * abs(line["losses"]["hint"])
        assert abs(float(dump["kd_loss"]) - line["losses"]["kd"]) <= 1e-6 * abs(line["losses"]["kd"])
        assert np.all(np.isfinite(dump["grads"])) and np.any(dump["grads"] != 0)
        dumps.append(dump)
    for name, a in dumps[0].items():
        np.testing.assert_allclose(dumps[1][name], a, rtol=1e-3, atol=1e-3 * float(np.abs(a).max()), err_msg=name)


def test_smem_floor_model():
    """roofline.smem_floor: DESIGN.md 4.0's shared-memory byte model applied to the default workload."""
    sys.path.insert(0, ROOT)
    import bench
    plan = bench.plan_51m()
    need_dx = [False] + [True] * (len(plan) - 1)
    planes = 4 * sum(ci for ci, _ in plan)
    f = bench.smem_floor(plan, 4, (9, 5, 20), "nchw", 128, need_dx, 2.66, 1900.0)
    want = ((planes - 4 * plan[0][0]) * 618 * 1024 + planes * 378 * 1024) / 128 / 148 / 1.9e6
    assert abs(f["ms"] - want) < 1e-3 and 0 < f["frac"] < 1
    assert bench.smem_floor(plan, 4, (9, 5, 20), "nhwc", 128, need_dx, 3.15, 1900.0) is None
    assert bench.smem_floor(plan, 4, (9, 5, 20), "nchw", 128, need_dx, 3.15, None) is None
    assert bench.smem_floor(plan, 4, (3, 1, 1), "nchw", 128, need_dx, 3.15, 1900.0) is None
