"""The tile-major step loop of ``k_fused_tma`` (``drsim_run_tape``, one launch per block of scheduled records): a CTA
runs each of its tiles through every step of the block before its next tile.  Bit for bit against one launch per
step (``DRSIM_NO_STREAM=1``) on the shapes the step-major loop it replaced could not take."""
import copy
import os

import pytest

pytestmark = pytest.mark.gpu

KEYS = ("dt_air", "dt_mass", "sso", "flags", "reward", "obs", "signal", "power", "od_temp", "metrics")


def _prop(n, **over):
    p = {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
         "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0},
                          "agents_comm_prop": {"max_nb_agents_communication": 10}},
         "power_grid_prop": {"signal_properties": {"mode": "sinusoidals"}}}
    for path, v in over.items():
        d = p
        keys = path.split("/")
        for k in keys[:-1]:
            d = d.setdefault(k, {})
        d[keys[-1]] = v
    return p


@pytest.mark.parametrize("n,R,layout,policy,T,pre,tiles_per_cta", [
    (1000, 400, "tarmac", "external", 70, 0, (1, 2)),              # between one and two tiles per CTA
    (1000, 100, "tarmac", "external", 70, 0, (0, 1)),              # at most one tile per CTA, action tape
    (1000, 640, "tarmac", "external", 100, 5, (2, 3)),             # starts mid-block, crosses the 64-step boundary
    (37, 17507, "tarmac", "external", 70, 0, (2, 3)),              # padded rows (N % 4 != 0), ragged last tile
    (1000, 640, "none", "external", 70, 0, (2, 3)),                # no observation rows
    (1000, 100, "tarmac", "deadband_bangbang", 70, 0, (0, 1))])    # on-device policy, at most one tile per CTA
def test_tile_major_loop_equals_per_step_launches(n, R, layout, policy, T, pre, tiles_per_cta):
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    a = BatchedEnv(_prop(n, **{"cluster_prop/house_prop/deadband": 0.4}), R, policy=policy, noise="philox", seed=7,
                   obs_layout=layout)
    a.reset()
    info = a.sim.fused_info()
    lo, hi = tiles_per_cta
    assert info["variant"] == "staged" and lo * info["grid"] < info["tiles"] <= hi * info["grid"], info
    planes = 3
    tape = None
    if policy == "external":
        tape = (torch.rand((planes, R, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) < 0.5).to(torch.uint8)
    for t in range(pre):
        a.step(None if tape is None else tape[t % planes])
    b = copy.deepcopy(a)
    launches0 = a.sim.launch_count
    a.run(T, tape, rotate=True)
    torch.cuda.synchronize()
    blocks = (pre + T + 63) // 64 - pre // 64          # 64-step schedule blocks the run touches
    assert a.sim.launch_count - launches0 <= 3 * blocks  # one step kernel (+ two schedule kernels) per block, not T launches
    os.environ["DRSIM_NO_STREAM"] = "1"
    try:
        b.run(T, tape, rotate=True)
    finally:
        del os.environ["DRSIM_NO_STREAM"]
    torch.cuda.synchronize()
    keys = [k for k in KEYS if a.state[k] is not None]   # (obs_layout "none": no observation plane)
    for k in keys:
        assert torch.equal(a.state[k], b.state[k]), k
    # the loop leaves the handle in a state ordinary steps continue from
    a.step(None if tape is None else tape[0]); b.step(None if tape is None else tape[0])
    torch.cuda.synchronize()
    for k in keys:
        assert torch.equal(a.state[k], b.state[k]), k
