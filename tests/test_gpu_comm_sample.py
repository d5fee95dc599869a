"""``random_sample`` neighbours drawn on the device (DRSIM_COMM_SAMPLE) on every step-kernel route, against the oracle.

A ``random_sample`` handle draws the neighbours of every row from a Philox stream keyed by (seed, global replica,
global house, draw), where the draw is the handle's step count as the rows see it.  The oracle is given the handle's
own table of the current draw (``neighbour_index()``, checked bit for bit against ``comm_sample_np``), so each case
checks the messages the kernels gathered as well as everything else the step writes.  Each route must be planned as
the same handle in ``random_fixed`` mode is: same variant, clusters per tile and launches per step.
"""
import copy

import numpy as np
import pytest

import comm_sample_np
from oracle_driver import ROUTES, OracleDriver, config, loop_launches, same_state
from test_gpu_oracle_routes import LOOP_ROUTE, T_STEPS

pytestmark = pytest.mark.gpu


class SampleDriver(OracleDriver):
    """The oracle reads the handle's current ``[R, N, c]`` draw, sliced to the picked replicas."""

    def _table(self):
        return self.env.neighbour_index().cpu().numpy()[self.picks]


def _env(p, R, precision="f32", layout="hand_engineered", path="auto", seed=21, obs_dtype="float32", rep_offset=0):
    from marl_demandresponse_b200 import BatchedEnv

    return BatchedEnv(p, R, precision=precision, obs_layout=layout, noise="philox", seed=seed, path=path,
                      obs_dtype=obs_dtype, rep_offset=rep_offset)


def _route(env):
    info = env.sim.fused_info()
    return info["variant"], info["envs_per_tile"], info["tiles"]


# route -> the neighbour counts it takes in rows of messages (odd c, and c = N - 1 on the 10-house routes; k_fused_direct
# has room for one message in its 16-column rows)
COUNTS = {
    "k_fused_tma<2>": [1, 3, 5], "k_fused_tma<0>/1-per-tile": [1, 3], "k_fused_tma<0>/3-per-tile": [2, 5],
    "k_fused_rows<staged>": [7, 10], "k_fused_rows<unstaged>": [9, 10], "general/rows-fallback": [9, 10],
    "k_fused/chunked": [3, 10], "k_fused_direct": [1], "k_small": [3, 9], "k_shard": [3, 10], "four-kernel": [1, 4],
    "k_fused_direct<double>": [3, 10], "k_fused<double>/chunked": [3, 9], "k_small_gen<double>": [5, 9],
    "k_shard<double>": [3, 10],
}
# the matrix cells the routes take (penalty etc.), as in test_gpu_oracle_routes
CELL = {"general/rows-fallback": dict(pen="common_L2"), "k_fused_tma<0>/1-per-tile": dict(pen="mixture", msg="th_hvac"),
        "k_fused_tma<0>/3-per-tile": dict(pen="common_max_error", state="solar"), "k_fused/chunked": dict(msg="th_hvac"),
        "k_small_gen<double>": dict(state="all", msg="th_hvac"), "k_fused_direct<double>": dict(pen="mixture"),
        "k_shard<double>": dict(state="solar"), "four-kernel": dict(pen="common_L2", state="solar")}
CASES = [pytest.param(r, c, id=f"{r}-c{c}") for r in COUNTS for c in COUNTS[r]]
TARMAC = [pytest.param(r, id=r) for r in ("k_fused_tma<1>", "k_fused_tma<0>/3-per-tile", "k_shard", "k_small")]


def _make(route, c, monkeypatch, layout=None, obs_dtype="float32", nb="random_sample"):
    precision, R, N, lay, path, env_vars, expect = ROUTES[route]
    layout = layout or lay
    for k, v in env_vars.items():
        monkeypatch.setenv(k, str(v))
    cell = dict(CELL.get(route, {}), sig="sinusoidals")
    p = config(N, nb=nb, c=c, **cell)
    return _env(p, R, precision, layout, path, obs_dtype=obs_dtype), p


def _check_route(route, env, p, layout, monkeypatch):
    """The route of the `random_fixed` twin, and the one the route table names."""
    precision, R, N, lay, path, env_vars, expect = ROUTES[route]
    c = env.comm_width
    twin, _ = _make(route, c, monkeypatch, layout=layout, nb="random_fixed")
    assert _route(env) == _route(twin), (_route(env), _route(twin))
    info = env.sim.fused_info()
    if "variant" in expect:
        assert info["variant"] == expect["variant"], info
    if "e" in expect:
        assert info["envs_per_tile"] == expect["e"], info
    return twin


def _run_against_oracle(env, p, R, N, seed, twin=None, launches=None, route=None):
    from marl_demandresponse_b200.batched import synthetic_state

    st = synthetic_state(p, R, seed=seed)
    env.reset(copy.deepcopy(st))
    if twin is not None:
        twin.reset(copy.deepcopy(st))
    drv = SampleDriver(env, p, st)
    drv.start_free()
    acts = (np.random.default_rng(seed).random((T_STEPS, R, N)) < 0.5).astype(np.uint8)
    got = []
    for t in range(T_STEPS):
        got.append(drv.step(acts[t]))
        if twin is not None:
            import torch

            l0 = twin.sim.launch_count
            twin.step(torch.as_tensor(acts[t], device="cuda"))
            assert got[-1] == twin.sim.launch_count - l0, ("launches", t)
            assert env.sim.last_route == twin.sim.last_route, t
        if route is not None and t == 0:
            assert env.sim.last_route == route, (env.sim.last_route, env.sim.fused_info())
    if launches is not None:
        assert got == [launches + 2] + [launches] * (T_STEPS - 1), got
    drv.check_metrics()
    drv.check_free()
    return drv


@pytest.mark.parametrize("route,c", CASES)
def test_route_matches_oracle(route, c, monkeypatch):
    """24 steps re-anchored and free-running against the oracle given the handle's own draws; same route and launches
    per step as a `random_fixed` twin."""
    env, p = _make(route, c, monkeypatch)
    twin = _check_route(route, env, p, ROUTES[route][3], monkeypatch)
    _run_against_oracle(env, p, env.n_replicas, env.n_houses, 40 + c, twin, ROUTES[route][6]["launches"],
                        ROUTES[route][6]["route"])
    # the rows' draw is the step count, and the handle's table is the NumPy restatement of it
    assert env.sim.step_count == T_STEPS
    want = comm_sample_np.comm_sample_table(env.seed, env.n_replicas, env.n_houses, T_STEPS, env.comm_width)
    assert np.array_equal(env.neighbour_index().cpu().numpy(), want)


@pytest.mark.parametrize("route,c", [p for p in CASES if ROUTES[p.values[0]][0] == "f32"])
def test_bf16_rows_are_the_fp32_rows_rounded(route, c, monkeypatch):
    import torch

    from marl_demandresponse_b200.batched import synthetic_state

    a, p = _make(route, c, monkeypatch)
    b, _ = _make(route, c, monkeypatch, obs_dtype="bfloat16")
    R, N = a.n_replicas, a.n_houses
    st = synthetic_state(p, R, seed=5)
    a.reset(copy.deepcopy(st))
    b.reset(copy.deepcopy(st))
    rng = np.random.default_rng(c)
    for t in range(6):
        acts = torch.as_tensor((rng.random((R, N)) < 0.5).astype(np.uint8), device="cuda")
        a.step(acts)
        b.step(acts)
        torch.cuda.synchronize()
        assert torch.equal(b.obs, a.obs.to(torch.bfloat16)), (route, t)
        assert torch.equal(a.reward, b.reward)


@pytest.mark.parametrize("route", TARMAC)
def test_tarmac_neighbour_index(route, monkeypatch):
    """No messages in the rows; neighbour_index() is the draw behind them."""
    env, p = _make(route, 10 if ROUTES[route][2] > 10 else 9, monkeypatch, layout="tarmac")
    _check_route(route, env, p, "tarmac", monkeypatch)
    _run_against_oracle(env, p, env.n_replicas, env.n_houses, 7, route=ROUTES[route][6]["route"])
    for d in (None, 0, 3, T_STEPS):
        want = comm_sample_np.comm_sample_table(env.seed, env.n_replicas, env.n_houses, T_STEPS if d is None else d, env.comm_width)
        assert np.array_equal(env.neighbour_index(d).cpu().numpy(), want), d


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_message_columns_are_the_records_of_the_drawn_houses(precision):
    """Every message column of every row equals the message record (norm.py:31-60) of the house the draw names."""
    from marl_demandresponse_b200.batched import synthetic_state

    R, N, c = 40, 100, 7
    p = config(N, nb="random_sample", c=c)
    env = _env(p, R, precision)
    env.reset(synthetic_state(p, R, seed=2))
    import torch

    for t in range(3):
        env.step(torch.as_tensor((np.random.default_rng(t).random((R, N)) < 0.5).astype(np.uint8), device="cuda"))
    torch.cuda.synchronize()
    s = env.get_state()
    cfg = env.sim.cfg
    obs = env.obs.double().cpu().numpy()
    tab = env.neighbour_index().cpu().numpy()
    assert np.array_equal(tab, comm_sample_np.comm_sample_table(env.seed, R, N, 3, c))
    msg = obs[..., 10:10 + 4 * c].reshape(R, N, c, 4)
    pmax = s["cap"] / cfg.cop / cfg.norm_reg_sig
    rec = np.stack([(s["t_air"] - s["target"]) / 5.0, (s["sso"] // cfg.lockout_duration).astype(np.float64),
                    s["on"] * pmax, pmax], axis=-1)                                   # [R, N, 4]
    gathered = np.take_along_axis(rec[:, None, :, :], tab[..., None].astype(np.int64), axis=2)   # [R, N, c, 4]
    tol = 1e-9 if precision == "f64" else 1e-5
    np.testing.assert_allclose(msg, gathered, rtol=tol, atol=tol)


# route, R, N, layout, environment, cell, steps before the run, run length
LOOP = [
    ("k_small", 7, 10, {}, dict(c=9), 0, 70),
    ("k_small", 5, 10, {}, dict(c=3, pen="mixture"), 5, 100),
    ("k_fused_tma<2>", 1800, 100, {"DRSIM_TILE_ENVS": 3}, dict(c=3), 0, 70),
    ("k_fused_tma<0>", 300, 300, {"DRSIM_TILE_ENVS": 1}, dict(c=3, pen="common_max_error", msg="th_hvac"), 5, 100),
    ("k_fused_tma<0>", 1800, 100, {"DRSIM_TILE_ENVS": 3}, dict(c=2, pen="mixture", state="all"), 0, 70),
    ("k_fused_rows", 4096, 100, {}, dict(c=10), 0, 70),
    ("k_fused_rows", 4096, 100, {}, dict(c=7), 5, 100),
]


@pytest.mark.parametrize("route,R,N,env_vars,cell,pre,T", [pytest.param(*c, id=f"{c[0]}-{i}") for i, c in enumerate(LOOP)])
def test_in_kernel_loop(route, R, N, env_vars, cell, pre, T, monkeypatch):
    """``run(T, tape, rotate=True)``: one step kernel per schedule block, the bits of one launch per step, and the
    free-running oracle given the handle's final draw; also from the middle of a block."""
    import torch

    from marl_demandresponse_b200.batched import synthetic_state

    for k, v in env_vars.items():
        monkeypatch.setenv(k, str(v))
    p = config(N, nb="random_sample", sig="sinusoidals", **cell)
    env = _env(p, R, seed=31)
    twin_fixed = _env(config(N, nb="random_fixed", sig="sinusoidals", **cell), R, seed=31)
    assert _route(env) == _route(twin_fixed)
    info = env.sim.fused_info()
    if route == "k_fused_rows":
        assert info["variant"] == "staged_rows" and min(info["grid"], info["tiles"] // 2) * 10 >= info["grid"] * 9, info
    elif route != "k_small":
        assert info["variant"] == "staged", info
    st = synthetic_state(p, R, seed=4)
    env.reset(copy.deepcopy(st))
    planes = 3
    tape = (torch.rand((planes, R, N), device="cuda", generator=torch.Generator(device="cuda").manual_seed(6)) < 0.5)
    tape = tape.to(torch.uint8)
    tape_np = tape.cpu().numpy()
    drv = SampleDriver(env, p, st)
    for t in range(pre):
        drv.step(tape_np[t % planes], check=False)
    twin = copy.deepcopy(env)
    drv.start_free()
    l0 = env.sim.launch_count
    env.run(T, tape, rotate=True)
    torch.cuda.synchronize()
    assert env.sim.last_route == LOOP_ROUTE.get(route, route), (env.sim.last_route, info)
    assert env.sim.launch_count - l0 == loop_launches(pre, T, 0 if pre else None)
    monkeypatch.setenv("DRSIM_NO_STREAM", "1")
    twin.run(T, tape, rotate=True)
    monkeypatch.delenv("DRSIM_NO_STREAM")
    torch.cuda.synchronize()
    same_state(env, twin)
    assert env.sim.step_count == pre + T == twin.sim.step_count
    for k in range(T):
        drv.advance_free(tape_np[k % planes])
    drv.check_free(f"{route}: run({T}) from step {pre}")


def test_replica_split_reproduces_one_handle():
    import torch

    from marl_demandresponse_b200.batched import synthetic_state

    R, N, c = 64, 100, 10
    p = config(N, nb="random_sample", c=c)
    st = synthetic_state(p, R, seed=8)
    whole = _env(p, R)
    halves = [_env(p, R // 2, rep_offset=o) for o in (0, R // 2)]
    whole.reset(copy.deepcopy(st))
    for h, o in zip(halves, (0, R // 2)):
        h.reset({k: (v[o:o + R // 2] if np.ndim(v) >= 1 and np.shape(v)[0] == R else v) for k, v in st.items()})
    rng = np.random.default_rng(1)
    for t in range(5):
        acts = torch.as_tensor((rng.random((R, N)) < 0.5).astype(np.uint8), device="cuda")
        whole.step(acts)
        for h, o in zip(halves, (0, R // 2)):
            h.step(acts[o:o + R // 2].contiguous())
        torch.cuda.synchronize()
        assert torch.equal(torch.cat([h.obs for h in halves]), whole.obs), t
        assert torch.equal(torch.cat([h.neighbour_index() for h in halves]), whole.neighbour_index()), t


def test_clone_continues_and_device_reset_restarts_the_draws():
    import torch

    from marl_demandresponse_b200.batched import synthetic_state

    R, N, c = 30, 100, 5
    p = config(N, nb="random_sample", c=c)
    env = _env(p, R)
    env.reset(synthetic_state(p, R, seed=3))
    rng = np.random.default_rng(2)
    acts = [torch.as_tensor((rng.random((R, N)) < 0.5).astype(np.uint8), device="cuda") for _ in range(6)]
    for a in acts[:3]:
        env.step(a)
    other = env.clone()
    assert other.sim.step_count == env.sim.step_count == 3
    for a in acts[3:]:
        env.step(a)
        other.step(a)
        torch.cuda.synchronize()
        assert torch.equal(env.obs, other.obs)
    assert torch.equal(env.neighbour_index(), other.neighbour_index())
    env.reset(device_mode="reference")
    torch.cuda.synchronize()
    assert env.sim.step_count == 0
    assert np.array_equal(env.neighbour_index().cpu().numpy(), comm_sample_np.comm_sample_table(env.seed, R, N, 0, c))
    env.step(acts[0])   # the reset's rows carry draw 0, the first step's rows draw 1
    torch.cuda.synchronize()
    assert env.sim.step_count == 1
    assert np.array_equal(env.neighbour_index().cpu().numpy(), comm_sample_np.comm_sample_table(env.seed, R, N, 1, c))


def test_collect_equals_policy_step_plus_step_and_buffer_tables():
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.rollout import RolloutBuffer

    R, N, c, T = 32, 100, 10, 6
    p = config(N, nb="random_sample", c=c)
    st = synthetic_state(p, R, seed=4)
    a, b = _env(p, R, seed=17), _env(p, R, seed=17)
    a.reset(copy.deepcopy(st))
    b.reset(copy.deepcopy(st))
    for e in (a, b):
        e.step(torch.zeros((R, N), dtype=torch.uint8, device="cuda"))   # collect from a handle that has stepped
    torch.manual_seed(3)
    fc = torch.nn.ModuleList([torch.nn.Linear(a.sim.D, 100), torch.nn.Linear(100, 100), torch.nn.Linear(100, 2)]).cuda()
    weights = BatchedEnv.actor_weights(fc)
    buf = RolloutBuffer(a, T)
    a.collect(weights, buf)
    assert buf.draw0 == 1
    for t in range(T):
        assert torch.equal(buf.state(t), b.obs), ("state", t)
        assert torch.equal(buf.neighbour_index(t), b.neighbour_index()), ("table", t)
        act, _ = b.policy_step(weights)
        assert torch.equal(buf.action(t), act), ("action", t)
        b.sim.step(None)
        assert torch.equal(buf.reward(t), b.reward), ("reward", t)
    assert torch.equal(buf.next_state(T - 1), b.obs)
    assert torch.equal(buf.neighbour_index(T), a.neighbour_index())
