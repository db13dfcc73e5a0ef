"""bench.py pieces that run without a GPU: the reference arm (`--impl reference`: the unmodified reference from
baseline/_ref, or the oracle port where that install is absent, timed on the host cores), its behaviour under a multi-rank launch, and the loud failure of the sm_100a arm on a box without a GPU."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, timeout=300, env=e, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    res = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--batch", "128"])
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("fused-pool fwd+bwd samples/sec at B=64K,M=3,D=512,H=8")
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    installed = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "aecf", "__init__.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if installed else "port") and d["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
    assert d["steps"] == 2 and d["warmup"] == 1 and d["same_config"] is True and "128 rows" in d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["tokens"] == 3 and d["config"]["embed_dim"] == 512 and d["config"]["heads"] == 8


def test_reference_arm_runs_on_rank_zero_only():
    res = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--batch", "64"],
               env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and not [l for l in res.stdout.splitlines() if l.startswith("{")]


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box without a GPU")
def test_b200_arm_fails_loudly_without_a_gpu():
    res = _run(["--steps", "1", "--warmup", "1", "--no-e2e", "--no-cpu-baseline"])
    assert res.returncode != 0 and "no CPU path" in res.stderr


def test_steps_below_one_are_refused():
    res = _run(["--steps", "0", "--warmup", "1"])
    assert res.returncode != 0 and "--steps" in res.stderr


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    res = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--batch", "64", "--dump-outputs", str(tmp_path / "d")])
    assert res.returncode != 0 and "--dump-outputs" in res.stderr and not os.path.exists(tmp_path / "d")


def test_dumped_outputs_are_a_fixed_float32_sample_within_the_budget(tmp_path):
    import numpy as np

    import bench
    torch.manual_seed(0)
    outputs = {"out": torch.randn(1000, 1, 64).bfloat16(), "grad_x": torch.randn(1000, 3, 64),
               "grad_w": torch.randn(48, 64), "entropy_loss": torch.tensor(0.25), "note": None}
    budget = 256 << 10
    a, b = bench.sample_outputs(outputs, budget), bench.sample_outputs(outputs, budget)
    assert set(a) == {"out", "grad_x", "grad_w", "entropy_loss"}
    assert sum(t.numel() * 4 for t in a.values()) <= budget
    assert all(t.dtype == torch.float32 and torch.equal(t, b[k]) for k, t in a.items())
    assert torch.equal(a["grad_w"], outputs["grad_w"]) and a["entropy_loss"].item() == 0.25     # small arrays whole
    for k in ("out", "grad_x"):                                  # too large: the first rows of a seeded permutation
        n = a[k].shape[0]
        assert 1 <= n < 1000 and a[k].shape[1:] == outputs[k].shape[1:]
        rows = torch.from_numpy(np.sort(np.random.default_rng(0).permutation(1000)[:n]))
        assert torch.equal(a[k], outputs[k][rows].float())
    bench.write_outputs(str(tmp_path), a)
    for k, t in a.items():
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, t.numpy())
