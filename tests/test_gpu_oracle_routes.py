"""Every step-kernel route, and the in-kernel step loop, against the fp64 NumPy oracle.

The step has one specification, ``oracle/np_oracle.py``, and many implementations; the host picks one from the
shape and the configuration (``plan_fused`` and ``step_route`` in ``drsim_api.cu``).  The routes: the four-kernel
path (``k_house`` + ``k_reduce`` + ``k_env`` + ``k_obs``), ``k_shard``, chunked ``k_fused``, ``k_fused_direct``,
``k_fused_tma<0|1|2>``, ``k_fused_rows<staged|unstaged>``, ``k_small`` and ``k_small_gen<double>``.  Each case below
names the route it means to run and fails if the host stops sending it there: ``last_route`` gives the kernels the
step ran on, ``fused_info()`` the tile variant and the clusters per tile, ``launch_count`` the launches per step.

* ``test_route_matches_oracle``: a mode matrix over the routes (a covering design, not the full product), 24 steps
  re-anchored on the oracle at every step, and the same steps free-running.
* ``test_seeded_sweep_matches_oracle``: random (R, N, layout, modes) from a fixed list of seeds.
* ``test_in_kernel_loop_matches_oracle``: ``run(T, tape, rotate=True)`` on the loop routes: one step kernel per
  schedule block, bit-identical to one launch per step, and free-running against the oracle.
* ``test_route_interpolation_matches_oracle``: every route with the interpolated base power, fired every third step
  (period 12 and 10 s: a multiple of the 4 s step and not) and on every step (period 3 s).  A firing step runs on
  ``k_shard`` (the four-kernel path where k_shard is off), the next step back on the route, after regenerating the
  schedule block the firing step ended.  The device's base power is checked against ``interp_ref`` at every firing,
  the reset's included.

Tolerances and the replicas compared are those of ``oracle_driver``.
"""
import copy
import os

import numpy as np
import pytest

from oracle_driver import NB_2D, ROUTES, OracleDriver, config, loop_launches, same_state

pytestmark = pytest.mark.gpu

T_STEPS = 24   # a 40 s lock-out is 10 steps of 4 s: lock-outs expire and re-arm within the run

# the mode matrix: every value of every axis on every route that can take it, plus penalty x clusters per tile
# (the k_fused_tma<0> routes with one and three clusters per tile), flags x odd D and neighbour mode x clusters per tile.
# Routes that cannot take a value: k_fused_tma<1|2> and k_fused_rows only run the individual penalty with plain rows
# (a common penalty there is the rows fallback / k_fused_tma<0>); k_small takes plain rows only.
MATRIX = {
    "k_fused_tma<1>": [dict(sig="perlin"), dict(sig="sinusoidals"), dict(sig="regular_steps"), dict(sig="flat"),
                       dict(sig="perlin", layout="hand_engineered", c=0)],
    "k_fused_tma<2>": [dict(sig="perlin", nb="neighbours", c=1), dict(sig="sinusoidals", nb="random_fixed", c=3),
                       dict(sig="regular_steps", nb="closed_groups", c=5), dict(sig="flat", nb="neighbours_2D", c=10)],
    "k_fused_tma<0>/1-per-tile": [
        dict(pen="common_L2", sig="perlin", nb="neighbours", c=1),
        dict(pen="common_max_error", sig="sinusoidals", state="solar", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", state="all", nb="closed_groups", c=5),
        dict(sig="flat", state="solar", nb="neighbours_2D"),
        dict(pen="mixture", sig="perlin", c=0),
        dict(pen="common_L2", sig="sinusoidals", state="solar", layout="tarmac")],
    "k_fused_tma<0>/3-per-tile": [
        dict(pen="common_L2", sig="perlin", nb="neighbours", c=2),
        dict(pen="common_max_error", sig="sinusoidals", state="solar", msg="th_hvac", nb="random_fixed", c=2),
        dict(pen="mixture", sig="regular_steps", state="all", nb="neighbours_2D"),
        dict(sig="flat", state="solar", nb="closed_groups", c=3),
        dict(pen="common_max_error", sig="flat", c=0),
        dict(sig="sinusoidals", layout="tarmac")],
    "k_fused_rows<staged>": [dict(sig="perlin", c=10), dict(sig="sinusoidals", nb="random_fixed", c=7),
                             dict(sig="regular_steps", nb="closed_groups", c=9), dict(sig="flat", nb="neighbours_2D", dist=2)],
    "k_fused_rows<unstaged>": [dict(sig="perlin", c=10), dict(sig="sinusoidals", nb="random_fixed", c=10),
                               dict(sig="regular_steps", nb="closed_groups", c=9), dict(sig="flat", nb="neighbours_2D", dist=2)],
    "general/rows-fallback": [dict(pen="common_L2", sig="perlin"), dict(pen="common_max_error", sig="sinusoidals", nb="random_fixed"),
                              dict(pen="mixture", sig="regular_steps", nb="closed_groups", c=9),
                              dict(pen="common_L2", sig="flat", nb="neighbours_2D", dist=2)],
    "k_fused/chunked": [
        dict(pen="common_L2", sig="perlin", state="solar", nb="neighbours", c=10),
        dict(pen="common_max_error", sig="sinusoidals", state="all", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", msg="th_hvac", nb="closed_groups", c=9),
        dict(sig="flat", state="solar", msg="th_hvac", nb="neighbours_2D"),
        dict(sig="perlin", state="all", msg="th_hvac", c=1)],
    "k_fused_direct": [   # (no room for message flags or a 2-D neighbourhood in rows of 16 columns)
        dict(pen="common_L2", sig="perlin", layout="tarmac"),
        dict(pen="common_max_error", sig="sinusoidals", state="solar", layout="tarmac"),
        dict(pen="mixture", sig="regular_steps", state="all", layout="tarmac"),
        dict(sig="flat", c=1),
        dict(pen="common_max_error", sig="perlin", nb="random_fixed", c=1),
        dict(pen="mixture", sig="sinusoidals", nb="closed_groups", c=1),
        dict(sig="regular_steps", state="solar", c=0)],
    "k_small": [dict(pen="common_L2", sig="perlin", c=9), dict(pen="common_max_error", sig="sinusoidals", nb="random_fixed", c=3),
                dict(pen="mixture", sig="regular_steps", nb="closed_groups", c=4), dict(sig="flat", c=0),
                dict(sig="perlin", c=1)],
    "k_shard": [
        dict(pen="common_L2", sig="perlin", c=10),
        dict(pen="common_max_error", sig="sinusoidals", state="solar", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", state="all", nb="closed_groups", c=10),
        dict(sig="flat", state="solar", nb="neighbours_2D"),
        dict(pen="mixture", sig="perlin", layout="tarmac"),
        dict(sig="sinusoidals", c=1), dict(pen="common_L2", sig="flat", c=0)],
    "four-kernel": [
        dict(pen="common_L2", sig="perlin", state="solar", c=1),
        dict(pen="common_max_error", sig="sinusoidals", state="all", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", msg="th_hvac", nb="closed_groups", c=10),
        dict(sig="flat", nb="neighbours_2D", c=0)],
    "k_fused_direct<double>": [
        dict(pen="common_L2", sig="perlin", c=10),
        dict(pen="common_max_error", sig="sinusoidals", state="solar", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", state="all", nb="closed_groups", c=4),
        dict(sig="flat", state="solar", nb="neighbours_2D"),
        dict(sig="perlin", c=1), dict(sig="sinusoidals", c=0)],
    "k_fused<double>/chunked": [
        dict(pen="common_L2", sig="perlin", c=10),
        dict(pen="common_max_error", sig="sinusoidals", state="all", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", state="solar", nb="closed_groups", c=9),
        dict(sig="flat", state="solar", msg="th_hvac", nb="neighbours_2D")],
    "k_small_gen<double>": [
        dict(pen="common_L2", sig="perlin", state="solar", c=9),
        dict(pen="common_max_error", sig="sinusoidals", state="all", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", msg="th_hvac", nb="closed_groups", c=4),
        dict(sig="flat", c=0), dict(sig="perlin", nb="neighbours_2D", n=12)],
    "k_shard<double>": [
        dict(pen="common_L2", sig="perlin", c=10),
        dict(pen="common_max_error", sig="sinusoidals", state="solar", msg="th_hvac", nb="random_fixed", c=3),
        dict(pen="mixture", sig="regular_steps", state="all", nb="closed_groups", c=10),
        dict(sig="flat", state="solar", nb="neighbours_2D"), dict(sig="sinusoidals", c=1)],
}
# neighbours_2D needs N % row_size == 0: the 10-house routes take it at N = 12 (its own case)
MATRIX["k_small"].append(dict(sig="perlin", nb="neighbours_2D", n=12, c=10))

CASES = [pytest.param(route, i, id=f"{route}-{i}") for route in ROUTES for i in range(len(MATRIX[route]))]


def _make(route, cell, monkeypatch, seed=21, table=None):
    """The handle of one matrix cell, its properties and initial state; asserts the route it takes."""
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    precision, R, N, layout, path, env_vars, expect = ROUTES[route]
    cell = dict(cell)
    layout = cell.pop("layout", layout)
    N = cell.pop("n", N)
    for k, v in env_vars.items():
        monkeypatch.setenv(k, str(v))
    p = config(N, **cell)
    env = BatchedEnv(p, R, precision=precision, obs_layout=layout, noise="philox", seed=seed, path=path, interp_table=table)
    info = env.sim.fused_info()
    print(route, cell, info)
    if "variant" in expect:
        assert info["variant"] == expect["variant"], (route, info)
    if "e" in expect:
        assert info["envs_per_tile"] == expect["e"], (route, info)
    st = synthetic_state(p, R, seed=seed + 1)
    env.reset(copy.deepcopy(st))
    return env, p, st, expect


@pytest.mark.parametrize("route,i", CASES)
def test_route_matches_oracle(route, i, monkeypatch):
    """24 steps of one matrix cell: every step re-anchored on the oracle (the single-step error), the trajectory
    free-running against the oracle, the running metrics, and the launches of each step."""
    env, p, st, expect = _make(route, MATRIX[route][i], monkeypatch)
    R, N = env.n_replicas, env.n_houses
    drv = OracleDriver(env, p, st)
    drv.start_free()
    acts = (np.random.default_rng(100 + i).random((T_STEPS, R, N)) < 0.5).astype(np.uint8)
    launches = [drv.step(acts[0])]
    assert env.sim.last_route == expect["route"], (route, MATRIX[route][i], env.sim.fused_info())
    launches += [drv.step(acts[t]) for t in range(1, T_STEPS)]
    # the first step generates the 64-step schedule block (two kernels), then one route's launches per step
    assert launches == [expect["launches"] + 2] + [expect["launches"]] * (T_STEPS - 1), launches
    drv.check_metrics()
    drv.check_free()


INTERP_PERIODS = [12, 10, 3]
INTERP_CASES = [pytest.param(route, period, id=f"{route}-interp{period}") for route in ROUTES for period in INTERP_PERIODS]


def interp_cell(cell, period, k=100):
    return {**cell, "power_grid_prop/base_power_props/mode": "interpolation",
            "power_grid_prop/base_power_props/interp_update_period": period,
            "power_grid_prop/base_power_props/interp_nb_agents": k}


def fire_schedule(period, T, dt=4):
    """Steps on which the interpolator fires after a reset that fired it (the counter starts at 0)."""
    c, out = 0, []
    for t in range(T):
        c += dt
        out.append(c >= period)
        if c >= period:
            c = 0
    return out


@pytest.mark.parametrize("route,period", INTERP_CASES)
def test_route_interpolation_matches_oracle(route, period, monkeypatch):
    """The first matrix cell of each route with the interpolated base power: re-anchored and free-running on the
    oracle, the routes and launches of firing steps, of the steps after them and of the schedule regeneration."""
    from oracle.config import synthetic_table

    table = synthetic_table(7)
    env, p, st, expect = _make(route, interp_cell(MATRIX[route][0], period), monkeypatch, table=table)
    R, N = env.n_replicas, env.n_houses
    drv = OracleDriver(env, p, st, table=table)
    got = env.get_state()
    assert np.all(got["t_since_interp"] == 0)            # the reset fired the interpolator
    drv.check_base_power(got, 0, "reset")
    drv.start_free()
    T = 12
    fires = fire_schedule(period, T)
    fire_route = "four-kernel" if "DRSIM_NO_SHARD_KERNEL" in ROUTES[route][5] else "k_shard"
    fire_launches = 4 if fire_route == "four-kernel" else 1
    acts = (np.random.default_rng(200 + period).random((T, R, N)) < 0.5).astype(np.uint8)
    valid = False   # the reset's refresh ended the schedule block
    for t in range(T):
        n = drv.step(acts[t])
        want_route = fire_route if fires[t] else expect["route"]
        want_n = (fire_launches if fires[t] else expect["launches"]) + (0 if valid else 2)
        assert (env.sim.last_route, n) == (want_route, want_n), (t, fires[t], env.sim.last_route, n, want_route, want_n)
        valid = not fires[t]
    assert drv.fired == [t for t in range(T) if fires[t]], drv.fired
    drv.check_metrics()
    drv.check_free()


@pytest.mark.parametrize("clear", ["set_state", "reset"])
@pytest.mark.parametrize("route", ["k_fused_tma<1>", "k_small", "k_small_gen<double>"])
def test_common_lockout_durations_restore_the_planned_route(route, clear, monkeypatch):
    """Per-house lock-out durations that differ take the general path; once they are common again (``set_state`` at
    the common duration, or a device reset) the handle is back on its planned route, with the bits of a fresh handle
    in the same state."""
    import torch

    env, p, st, expect = _make(route, MATRIX[route][0], monkeypatch)
    R, N = env.n_replicas, env.n_houses
    info = env.sim.fused_info()
    dur = int(env.sim.cfg.lockout_duration)
    rng = np.random.default_rng(3)
    mixed = np.full((R, N), dur, dtype=np.int32)
    mixed[:, ::2] = 2 * dur
    env.set_state({"lockout_duration": mixed})
    env.step(torch.as_tensor((rng.random((R, N)) < 0.5).astype(np.uint8), device="cuda"))
    assert env.sim.last_route in ("k_shard", "four-kernel"), env.sim.last_route
    assert env.sim.fused_info()["variant"] == "none"
    if clear == "set_state":
        env.set_state({"lockout_duration": np.full((R, N), dur, dtype=np.int32)})
    else:
        env.reset(device_mode="synthetic")
    assert env.sim.fused_info() == info
    fresh = copy.deepcopy(env)
    for t in range(3):
        acts = torch.as_tensor((rng.random((R, N)) < 0.5).astype(np.uint8), device="cuda")
        env.step(acts)
        fresh.step(acts)
        torch.cuda.synchronize()
        assert env.sim.last_route == fresh.sim.last_route == expect["route"], (t, env.sim.last_route)
        same_state(env, fresh)


SWEEP_SEEDS = list(range(20))


@pytest.mark.parametrize("seed", SWEEP_SEEDS)
def test_seeded_sweep_matches_oracle(seed):
    """Random (R, N, layout, modes) on whatever route the planner picks, re-anchored on the oracle at every step."""
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    rng = np.random.default_rng(1000 + seed)
    N = int(rng.choice([1, 2, 3, 5, 9, 10, 12, 33, 64, 100, 127, 128, 250, 300, 333, 512, 1000, 1023, 1024, 1300]))
    R = int(rng.integers(1, max(2, min(3000, 300000 // N))))
    layout = str(rng.choice(["tarmac", "hand_engineered", "none"]))
    precision = str(rng.choice(["f32", "f64"], p=[0.7, 0.3]))
    c = int(rng.choice([0, 1, 3, 4, 10, 11]))
    nb = str(rng.choice(["neighbours", "random_fixed", "closed_groups", "neighbours_2D"]))
    # (closed_groups: a last group one house short makes the reference's table point past the cluster)
    if nb == "neighbours_2D" and N not in NB_2D or nb == "closed_groups" and (c > N - 1 or N % (c + 1) == c):
        nb = "neighbours"
    cell = dict(pen=str(rng.choice(["individual_L2", "common_L2", "common_max_error", "mixture"])),
                sig=str(rng.choice(["perlin", "sinusoidals", "regular_steps", "flat"])),
                state=str(rng.choice(["none", "solar", "all"])), msg=str(rng.choice(["none", "th_hvac"])), nb=nb, c=c)
    # the base-power mode from a stream of its own (the draws above are those of the constant-power sweep)
    brng = np.random.default_rng(2000 + seed)
    table = None
    if brng.random() < 0.5:
        from oracle.config import synthetic_table

        table = synthetic_table(7)
        cell = interp_cell(cell, int(brng.choice([3, 10, 12, 40])), int(brng.choice([1, 10, 100])))
    p = config(N, **cell)
    env = BatchedEnv(p, R, precision=precision, obs_layout=layout, noise="philox", seed=seed, interp_table=table)
    print(seed, R, N, layout, precision, cell, env.sim.fused_info())
    st = synthetic_state(p, R, seed=seed)
    env.reset(copy.deepcopy(st))
    drv = OracleDriver(env, p, st, table=table)
    if table is not None:
        drv.check_base_power(env.get_state(), 0, "reset")
    T = 12
    acts = (rng.random((T, R, N)) < 0.5).astype(np.uint8)
    for t in range(T):
        drv.step(acts[t])
    drv.check_metrics()


# route, R, N, layout, environment, cell, steps before the run, run length, expected (fp32: the loop is fp32 only)
LOOP_CASES = [
    ("k_small", 7, 10, "hand_engineered", {}, dict(c=9), 0, 70, dict()),
    ("k_small", 7, 10, "hand_engineered", {}, dict(pen="common_max_error", nb="closed_groups", c=4, sig="sinusoidals"), 5, 100,
     dict()),
    ("k_small", 5, 10, "hand_engineered", {}, dict(pen="mixture", nb="random_fixed", c=3, sig="flat",
                                                   start="2021-12-31T23:58:20"), 0, 70, dict()),
    ("k_fused_tma<1>", 400, 1000, "tarmac", {}, dict(sig="perlin", start="2021-06-15T23:58:20"), 0, 70,
     dict(variant="staged", e=1)),
    ("k_fused_tma<1>", 640, 1000, "tarmac", {}, dict(sig="sinusoidals"), 5, 100, dict(variant="staged", e=1)),
    ("k_fused_tma<2>", 1800, 100, "hand_engineered", {"DRSIM_TILE_ENVS": 3}, dict(c=2, sig="regular_steps", nb="random_fixed",
                                                                                 start="2021-12-31T23:58:20"), 0, 70,
     dict(variant="staged", e=3)),
    ("k_fused_tma<0>", 400, 1000, "tarmac", {}, dict(pen="common_L2", state="solar", start="2021-12-31T23:58:20"), 0, 70,
     dict(variant="staged", e=1)),
    ("k_fused_tma<0>", 300, 300, "hand_engineered", {"DRSIM_TILE_ENVS": 1},
     dict(pen="common_max_error", state="solar", msg="th_hvac", nb="closed_groups", c=3, sig="sinusoidals"), 5, 100,
     dict(variant="staged", e=1)),
    ("k_fused_tma<0>", 1800, 100, "hand_engineered", {"DRSIM_TILE_ENVS": 3},
     dict(pen="mixture", state="all", nb="neighbours_2D", sig="perlin", start="2021-06-15T23:58:20"), 0, 70,
     dict(variant="staged", e=3)),
    ("k_fused_tma<0>", 6100, 100, "tarmac", {}, dict(pen="common_max_error", sig="flat"), 5, 100,
     dict(variant="staged")),
    ("k_fused_rows", 4096, 100, "hand_engineered", {}, dict(c=10, sig="sinusoidals", start="2021-06-15T23:58:20"), 0, 70,
     dict(variant="staged_rows")),
    ("k_fused_rows", 4096, 100, "hand_engineered", {}, dict(c=10, nb="random_fixed", sig="perlin"), 5, 100,
     dict(variant="staged_rows")),
]


# the loop takes k_fused_rows in its staged variant only
LOOP_ROUTE = {"k_fused_rows": "k_fused_rows<staged>"}


@pytest.mark.parametrize("route,R,N,layout,env_vars,cell,pre,T,expect",
                         [pytest.param(*c, id=f"{c[0]}-{i}") for i, c in enumerate(LOOP_CASES)])
def test_in_kernel_loop_matches_oracle(route, R, N, layout, env_vars, cell, pre, T, expect, monkeypatch):
    """``run(T, tape, rotate=True)`` with the step loop inside the kernel: one step kernel per schedule block, the same
    bits as one launch per step (``DRSIM_NO_STREAM=1``), and the trajectory free-running against the oracle."""
    import datetime as _dt

    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    for k, v in env_vars.items():
        monkeypatch.setenv(k, str(v))
    p = config(N, **cell)
    env = BatchedEnv(p, R, obs_layout=layout, noise="philox", seed=31)
    info = env.sim.fused_info()
    print(route, cell, info)
    for k in ("variant", "e"):
        if k in expect:
            assert info[{"e": "envs_per_tile"}.get(k, k)] == expect[k], info
    if route == "k_fused_rows":   # the loop takes k_fused_rows on at least two tiles per CTA (the `taped` condition)
        assert (min(info["grid"], info["tiles"] // 2)) * 10 >= info["grid"] * 9, info
    start = _dt.datetime.fromisoformat(cell["start"]) if "start" in cell else None
    st = synthetic_state(p, R, seed=4, start=start)
    env.reset(copy.deepcopy(st))
    planes = 3
    tape = (torch.rand((planes, R, N), device="cuda", generator=torch.Generator(device="cuda").manual_seed(6)) < 0.5)
    tape = tape.to(torch.uint8)
    tape_np = tape.cpu().numpy()
    drv = OracleDriver(env, p, st)
    for t in range(pre):
        drv.step(tape_np[t % planes], check=False)
    twin = copy.deepcopy(env)
    drv.start_free()
    l0 = env.sim.launch_count
    env.run(T, tape, rotate=True)
    torch.cuda.synchronize()
    assert env.sim.last_route == LOOP_ROUTE.get(route, route), (env.sim.last_route, info)
    # (the first of the steps before the run generated the block that starts at step 0; set_state invalidates it)
    assert env.sim.launch_count - l0 == loop_launches(pre, T, 0 if pre else None), (env.sim.launch_count - l0, pre, T)
    monkeypatch.setenv("DRSIM_NO_STREAM", "1")
    twin.run(T, tape, rotate=True)
    monkeypatch.delenv("DRSIM_NO_STREAM")
    torch.cuda.synchronize()
    same_state(env, twin)
    for k in range(T):
        drv.advance_free(tape_np[k % planes])
    drv.check_free(f"{route}: run({T}) from step {pre}")
