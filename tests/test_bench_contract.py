"""bench.py contract checks: the reference arm prints ONE JSON line with the keys a caller reads, non-zero ranks of a
multi-process launch exit without work, the GPU arm refuses to run without a device, and `--dump-outputs` writes the
headline's last step within its size budget, the same arrays every run (on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          env=e, timeout=timeout, cwd=ROOT)


def test_reference_arm_line():
    # small grid / 2 frames so that the CPU port finishes in seconds; the default run uses grid 64 and a full clip
    p = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--grid", "32", "--points", "2000",
              "--cpu-baseline-frames", "2"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    # kind = "reference" when oracle/_ref holds the staged reference (build container / GPU box), else the oracle port
    assert d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    # the line says what actually ran: one timed step of ONE clip x 2 frames, not the GPU arm's 64-clip step
    assert d["steps"] == 1 and d["warmup"] == 1 and d["config"]["clips_per_step"] == 1 and d["config"]["frames_per_clip"] == 2
    assert abs(d["value"] - 2 / (d["ms_per_step"] / 1e3)) <= 1e-6 * d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype"):
        assert k in d


def test_reference_arm_other_ranks_exit_quietly():
    p = _run(["--impl", "reference", "--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, timeout=120)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    p = _run(["--steps", "1"], timeout=300)
    assert p.returncode != 0 and "needs a GPU" in (p.stderr + p.stdout)


def test_steps_below_one_are_rejected():
    p = _run(["--impl", "reference", "--steps", "0"], timeout=120)
    assert p.returncode != 0 and "--steps" in p.stderr


def test_dump_outputs_is_rejected_for_the_reference_arm(tmp_path):
    p = _run(["--impl", "reference", "--dump-outputs", str(tmp_path / "d")], timeout=120)
    assert p.returncode != 0 and "--dump-outputs" in p.stderr and not (tmp_path / "d").exists()


def test_sample_outputs_keeps_the_budget_and_fixed_positions(tmp_path):
    import bench
    out = {"big": torch.arange(5_000_000, dtype=torch.float32), "kp": torch.rand(2, 3, 24, 4).half(),
           "idx": torch.arange(10, dtype=torch.int32), "loss": torch.tensor(0.25, dtype=torch.float64), "A_hats": None}
    got = bench.sample_outputs(out)
    assert sorted(got) == ["big", "idx", "kp", "loss"]
    assert sum(a.nbytes for _, a in got.values()) <= bench.DUMP_BYTES
    shape, big = got["big"]
    assert shape == [5_000_000] and big.dtype == np.float32 and big.size == bench.DUMP_BYTES // (8 * 4)
    assert np.all(np.diff(big) > 0) and big[-1] < 5_000_000              # distinct positions, in order
    assert np.array_equal(bench.sample_outputs(out)["big"][1], big)      # the same positions every call
    assert got["kp"][1].shape == (2, 3, 24, 4) and np.array_equal(got["kp"][1], out["kp"].float().numpy())
    assert got["idx"][1].dtype == np.float64 and got["loss"][1].dtype == np.float64 and got["loss"][1] == 0.25
    rec = bench.write_outputs(str(tmp_path / "dump"), got)
    assert rec["arrays"]["big"] == {"shape": [5_000_000], "saved": big.size}
    assert np.array_equal(np.load(tmp_path / "dump" / "big.npy"), big)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["detector", "generate"])
def test_dump_outputs_are_the_same_every_run(tmp_path, workload):
    args = ["--steps", "2", "--warmup", "1", "--clips", "2", "--frames", "7", "--points", "2000", "--grid", "32",
            "--workload", workload, "--no-sub", "--no-cpu-baseline"]
    runs = []
    for i in range(2):
        p = _run(args + ["--dump-outputs", str(tmp_path / str(i))])
        assert p.returncode == 0, p.stderr[-3000:]
        line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2
        runs.append(line["outputs"]["arrays"])
    assert runs[0] == runs[1] and "keypoints" in runs[0]
    kp = np.load(tmp_path / "0" / "keypoints.npy")                    # stored whole: (clips, frames, 24 joints, xyz + I)
    assert kp.shape == (2, 7, 24, 4) and np.isfinite(kp).all() and np.abs(kp).max() > 0
    files = sorted(os.listdir(tmp_path / "0"))
    assert files == sorted(f"{name}.npy" for name in runs[0])
    assert sum(os.path.getsize(tmp_path / "0" / f) for f in files) <= 64 << 20
    for f in files:
        a, b = np.load(tmp_path / "0" / f), np.load(tmp_path / "1" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b, equal_nan=True), f
