"""Host-side helpers of bench.py that do not need a GPU."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_usable_cores_respects_affinity_and_is_bounded():
    b = _bench()
    n = b.usable_cores()
    assert 1 <= n <= 32
    if hasattr(os, "sched_getaffinity"):
        assert n <= len(os.sched_getaffinity(0))


def test_cpu_samples_are_valid_configs():
    """Every bounded sample must be a config the discriminator accepts (side >= 128, divisible by 32) and ordered largest first."""
    b = _bench()
    costs = [side * side * t for side, t in b.CPU_SAMPLES]
    assert costs == sorted(costs, reverse=True)
    for side, t in b.CPU_SAMPLES:
        assert side >= 128 and side % 32 == 0 and t >= 1


def test_reference_arm_other_ranks_exit_silently():
    """Under torchrun only rank 0 runs the reference arm; the other ranks print nothing and exit 0 (bench contract)."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_writes_float32_and_a_fixed_sample_of_large_arrays(tmp_path, monkeypatch):
    """--dump-outputs: one float32 .npy per returned array, parameter samples for a training step, arrays over the cap sampled the
    same way on every run."""
    import numpy as np
    import torch

    b = _bench()
    monkeypatch.setattr(b, "DUMP_MAX_ELEMS", 100)
    monkeypatch.setattr(b, "DUMP_PARAM_SAMPLE", 50)
    nets = (torch.nn.Linear(8, 8), torch.nn.Linear(4, 2))
    outs = {"d_loss": torch.tensor(1.5), "out": torch.arange(300, dtype=torch.float64).reshape(3, 100)}
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), outs, nets)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert sorted(got) == ["d_loss", "discriminator_params", "generator_params", "out"]
    assert all(v.dtype == np.float32 for v in got.values())
    assert got["d_loss"].shape == () and float(got["d_loss"]) == 1.5
    assert got["out"].shape == (100,) and len(set(got["out"].tolist())) == 100
    assert got["generator_params"].shape == (50,) and got["discriminator_params"].shape == (10,)
    for name, v in got.items():
        assert np.array_equal(v, np.load(tmp_path / "b" / f"{name}.npy")), name


def test_flop_model_matches_design():
    """DESIGN.md section 4: one step = B * [2 (F_G + 6 F_D) + K (3 F_G + 3 F_D)] with F_G = 521.4 GF, F_D = 35.7 GF."""
    b = _bench()
    got = b.flop_step(16, 1)
    assert abs(got / 1e12 - 50.3) < 0.5, got
