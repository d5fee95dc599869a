"""bench.py's JSON contract, checked on the arm that runs without a GPU (``--impl reference``: the CPU
port of the reference step on all host cores) and on the argument parser of the GPU arm; ``--dump-outputs``."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=240, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    z = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in z, k
    assert z["impl"] == "reference" and z["metric"] == "house-steps/sec" and z["unit"] == "house-steps/s"
    assert z["higher_is_better"] is True and z["vs_baseline"] is None and z["value"] > 0
    assert z["config"]["workload"].startswith("C4")              # the configuration the metric is quoted on
    cb = z["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == z["value"] and cb["sample"]
    assert z["e2e"] == {"value": z["value"], "unit": z["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_under_torchrun_env_only_rank0_prints():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_samples_the_same_agents_in_every_file(tmp_path):
    import torch

    from bench import dump_outputs

    g = torch.Generator().manual_seed(0)
    obs = torch.rand((8, 50, 3), generator=g)
    arrays = {"obs": obs, "reward": obs.sum(-1), "power": obs[..., 0].double()}
    dump_outputs(str(tmp_path / "full"), arrays)
    assert np.load(tmp_path / "full" / "obs.npy").dtype == np.float32
    assert np.array_equal(np.load(tmp_path / "full" / "obs.npy"), obs.numpy())
    assert np.load(tmp_path / "full" / "power.npy").dtype == np.float64
    budget = 4000
    for d in ("a", "b"):
        dump_outputs(str(tmp_path / d), arrays, budget=budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["obs.npy", "power.npy", "reward.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= budget
    z = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    k = z["reward"].shape[0]
    assert 0 < k < 8 * 50 and z["obs"].shape == (k, 3) and z["power"].shape == (k,)
    np.testing.assert_array_equal(z["reward"], z["obs"].sum(-1, dtype=np.float32))
    rows = obs.reshape(-1, 3).numpy()
    assert all((rows == r).all(axis=1).any() for r in z["obs"])       # every kept row is an agent of the input
    for f in files:                                                  # the sample is fixed: identical files
        assert np.array_equal(z[f[:-4]], np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_dump_outputs_is_reproducible_and_steps_is_the_timed_count(tmp_path):
    out = {}
    for run in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "7", "--warmup", "2",
                              "--no-cpu", "--no-rollout", "--no-c5", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        z = json.loads([ln for ln in res.stdout.splitlines() if ln.strip()][-1])
        assert z["steps"] == 7
        out[run] = {f: np.load(tmp_path / run / (f + ".npy")) for f in ("obs", "reward")}
        assert sum(os.path.getsize(tmp_path / run / (f + ".npy")) for f in out[run]) <= 64_000_000
        assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in out[run].values())
    k = out["a"]["reward"].shape[0]
    assert out["a"]["obs"].shape == (k, 10) and k < 2048 * 1000   # C4 (D = 10) is over the budget: a sample of agents
    for f in out["a"]:
        np.testing.assert_allclose(out["b"][f], out["a"][f], rtol=1e-6, atol=1e-6)


@pytest.mark.gpu
def test_timed_region_runs_exactly_steps_environment_steps():
    """Every step advances each replica's clock by the time step: two device-resident runs that differ only in
    ``steps`` must advance it by exactly the difference (warm-up and pre-roll are the same in both)."""
    import argparse

    from bench import GpuWorkload

    w = GpuWorkload("c4", argparse.Namespace(exchange="peer", flush_l2=False), 0, 1, 0)
    advance = {}
    for steps in (7, 20):
        e0 = w.env.state["epoch"].clone()
        _, _, one_call = w.device_resident(steps, 2)
        assert one_call
        advance[steps] = (w.env.state["epoch"] - e0).cpu().numpy()
    dt = 4   # bench.env_prop_for: time_step 4 s
    assert ((advance[20] - advance[7]) == (20 - 7) * dt).all(), (advance[7][:4], advance[20][:4])
