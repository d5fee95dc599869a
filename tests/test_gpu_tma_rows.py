"""Observation rows of ``k_fused_tma<1>`` (one 10-column TarMAC row per house, one cluster per tile) on ragged clusters:
N % 4 in {1, 2, 3}, so the last thread of every tile holds one to three padding slots, with per-house targets that
differ from tile to tile, in fp32 and bf16.  The in-kernel step loop against one launch per step bit for bit, and both
against the four-kernel path (discrete state bit for bit, rows to the rounding of the cluster power)."""
import copy
import os
from contextlib import contextmanager

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ("dt_air", "dt_mass", "sso", "flags", "reward", "obs_padded", "signal", "power", "od_temp", "metrics")


def _prop(n):
    return {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
            "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0, "deadband": 0.4}},
            "power_grid_prop": {"signal_properties": {"mode": "sinusoidals"}}}


@contextmanager
def _env_var(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", [1001, 1002, 1003])
def test_ragged_rows_loop_launches_and_four_kernel_path(n, dtype):
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    R, T, planes = 700, 70, 3
    prop = _prop(n)
    st = synthetic_state(prop, R, seed=5)
    assert np.unique(st["target"][:, 0]).size == R   # per-house targets differ from replica (tile) to replica
    tape = (torch.rand((planes, R, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(6)) < 0.5)
    tape = tape.to(torch.uint8)

    a = BatchedEnv(prop, R, obs_layout="tarmac", noise="philox", seed=11, obs_dtype=dtype)
    a.reset(copy.deepcopy(st))
    info = a.sim.fused_info()
    assert info["variant"] == "staged" and info["envs_per_tile"] == 1 and info["tiles"] > info["grid"], info
    b = copy.deepcopy(a)
    a.run(T, tape, rotate=True)
    assert a.sim.last_route == "k_fused_tma<1>", a.sim.last_route
    with _env_var(DRSIM_NO_STREAM=1):
        b.run(T, tape, rotate=True)
    assert b.sim.last_route == "k_fused_tma<1>", b.sim.last_route
    torch.cuda.synchronize()
    for k in KEYS:
        assert torch.equal(a.state[k], b.state[k]), k
    assert not a.state["obs_padded"][:, n:, :].any()   # padding rows are zero

    with _env_var(DRSIM_NO_SHARD_KERNEL=1):
        c = BatchedEnv(prop, R, obs_layout="tarmac", noise="philox", seed=11, obs_dtype=dtype, path="split")
    c.reset(copy.deepcopy(st))
    with _env_var(DRSIM_NO_SHARD_KERNEL=1):
        c.run(T, tape, rotate=True)
    assert c.sim.last_route == "four-kernel", c.sim.last_route
    torch.cuda.synchronize()
    for k in ("dt_air", "dt_mass", "sso", "flags", "signal", "od_temp"):
        assert torch.equal(a.state[k], c.state[k]), k
    tol = 2e-6 if dtype == "float32" else 8e-3
    x, y = a.state["obs_padded"].float(), c.state["obs_padded"].float()
    torch.testing.assert_close(x, y, rtol=tol, atol=tol)
    # every column but the cluster power (column 4) is computed from the house alone: bit for bit
    keep = [q for q in range(10) if q != 4]
    assert torch.equal(a.state["obs_padded"][..., keep], c.state["obs_padded"][..., keep])
    torch.testing.assert_close(a.state["reward"], c.state["reward"], rtol=2e-6, atol=2e-6)
