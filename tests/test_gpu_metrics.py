"""The running metrics on the paths the oracle-driven route tests do not reach, and ``ReferenceMetrics`` at every shape.

* The six sums every step kernel keeps (``state["metrics"]``) against ``oracle_driver.metric_increments`` of the
  device's own planes, on every replica: steps with injected noise and steps where the interpolator fires (the inline
  epilogue), with junk in the padding slots of the temperature plane.
* Refreshes add nothing; a reset that starts an episode zeroes the sums, ``set_state`` keeps them.
* ``distributed.reduce_rollout_metrics`` against the restated sums, and replica-sharded handles against one handle.
* ``ReferenceMetrics`` (``k_metrics_ref``) against ``oracle.metrics_ref.BatchedRefMetrics`` fed the same planes, in
  both builds, one to 300 replicas, 10 to 2500 houses, padded rows, ``reset`` / ``initialize`` / ``log_values`` /
  ``rms``, and its refusal on a house-sharded handle.
"""
import numpy as np
import pytest

from oracle_driver import (check_metric_delta, metric_increments, metric_tolerance, own_plane_tolerance, prop, step_planes,
                           tolerances)

pytestmark = pytest.mark.gpu

PADDING_JUNK = 3.0   # deviation planted in the padding slots: a sum that is not masked picks it up


def _env(n, R, precision, **kw):
    from marl_demandresponse_b200 import BatchedEnv

    return BatchedEnv(kw.pop("env_prop", prop(n)), R, precision=precision, noise="philox", seed=9, **kw)


def _plant_padding(env):
    """Write ``PADDING_JUNK`` Ta - target into the padding slots ``[N, Ns)`` of every replica (none when N = Ns).  Some
    kernels store zeros there, so the junk is planted again before each step."""
    import torch

    v = env.state
    R, N, Ns = env.sim.R, env.sim.N, env.sim.Ns
    key = "dt_air" if v["temp_is_deviation"] else "t_air"
    full = v[key].as_strided((R, Ns), (Ns, 1))
    if not v["temp_is_deviation"]:   # fp64: absolute temperatures against the padding's set-point
        full[:, N:] = v["target"].as_strided((R, Ns), (Ns, 1))[:, N:] + PADDING_JUNK
    else:
        full[:, N:] = PADDING_JUNK
    torch.cuda.synchronize()


def _reset_across_target(env, seed=3):
    """The seeded synthetic state with every other replica moved 3 degrees down, so that some clusters start with
    a negative mean offset (a lost absolute value shows) and some with a positive one."""
    from marl_demandresponse_b200.batched import synthetic_state

    st = synthetic_state(env.props, env.n_replicas, seed, env.rep_offset)
    for k in ("t_air", "t_mass"):
        st[k][1::2] -= 3.0
    env.reset(st)
    _plant_padding(env)


def _metrics(env):
    import torch

    torch.cuda.synchronize()
    return env.state["metrics"].double().cpu().numpy()


def _precision(env):
    return "f64" if env.sim.real == np.float64 else "f32"


def _checked(env, step, what):
    """Plant junk in the padding slots, run ``step()`` (one environment step) and check what it added to the running
    metrics on every replica against the restatement from the planes before and after it.  Returns the restated
    increments and their tolerance."""
    _plant_padding(env)
    signal_before = env.get_state(["signal"])["signal"]
    m0 = _metrics(env)
    step()
    after = step_planes(env)
    m1 = _metrics(env)
    delta = m1 - m0
    precision = _precision(env)
    rel, p_rel = own_plane_tolerance(precision)
    want = metric_increments(signal_before, after)
    tol = metric_tolerance(signal_before, after, rel, p_rel, rew_rel=tolerances(precision, True)["rel"])
    check_metric_delta(delta, want, tol, what, sums=(m0, m1))
    return want, tol


def _acts(rng, R, n):
    import torch

    return torch.as_tensor((rng.random((R, n)) < 0.5).astype(np.uint8), device="cuda")


# ---- the inline epilogue -------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("n,R", [(10, 7), (37, 5), (1001, 3)])
def test_steps_with_injected_noise(precision, n, R):
    """Injected outdoor-temperature and Perlin noise leave the schedule: the step ends in the inline epilogue."""
    import torch

    env = _env(n, R, precision)
    _reset_across_target(env)
    rng = np.random.default_rng(1)
    for t in range(5):
        od = torch.as_tensor(rng.normal(size=R), device="cuda")
        pe = torch.as_tensor(rng.uniform(-1.0, 1.0, size=R), device="cuda")
        a = _acts(rng, R, n)
        _checked(env, lambda: env.step(a, od_noise=od, perlin=pe), f"{precision} N={n} injected noise, step {t}")


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("n,R,layout", [(101, 6, "hand_engineered"), (1000, 3, "tarmac")])
def test_steps_where_the_interpolator_fires(precision, n, R, layout):
    """Base power by interpolation, refreshed every third step: those steps end in the inline epilogue, the others
    on the route's own."""
    from oracle.config import synthetic_table

    p = prop(n, **{"power_grid_prop/base_power_props/mode": "interpolation",
                   "power_grid_prop/base_power_props/interp_update_period": 12})
    env = _env(n, R, precision, env_prop=p, obs_layout=layout, interp_table=synthetic_table(7))
    _reset_across_target(env)
    rng = np.random.default_rng(2)
    for t in range(10):
        a = _acts(rng, R, n)
        _checked(env, lambda: env.step(a), f"{precision} N={n} interpolation, step {t} ({env.sim.last_route})")


@pytest.mark.parametrize("route,cell", [("k_fused_direct", dict(pen="common_L2", layout="tarmac")),
                                        ("k_small", dict(pen="common_L2", c=9)), ("k_small_gen<double>", dict(c=9))])
def test_padded_routes(route, cell, monkeypatch):
    """The routes of the oracle route table whose clusters have padding slots (a cell of each that the route takes),
    each step checked on every replica with junk in the padding."""
    from oracle_driver import ROUTES, config

    precision, R, n, layout, path, environ, expected = ROUTES[route]
    assert n % 4, route
    cell = dict(cell)
    layout = cell.pop("layout", layout)
    for k, v in environ.items():
        monkeypatch.setenv(k, str(v))
    env = _env(n, R, precision, env_prop=config(n, **cell), obs_layout=layout, path=path)
    _reset_across_target(env)
    rng = np.random.default_rng(8)
    for t in range(4):
        a = _acts(rng, R, n)
        _checked(env, lambda: env.step(a), f"{route}, step {t}")
        assert env.sim.last_route == expected["route"], env.sim.last_route


# ---- refreshes and resets ------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("n,R", [(10, 7), (100, 30)])
def test_refreshes_add_nothing_and_resets_start_from_zero(precision, n, R):
    from marl_demandresponse_b200.batched import synthetic_state

    env = _env(n, R, precision)
    rng = np.random.default_rng(3)

    def run(k):
        for _ in range(k):
            env.step(_acts(rng, R, n))
        m = _metrics(env)
        assert np.all(m[:, 0] == k) and np.all(m[:, 4] > 0), m
        return m

    env.reset()
    m = run(3)
    env.sim.refresh(True)
    assert np.array_equal(_metrics(env), m), "a refresh changed the running metrics"
    env.set_state(env.get_state(["signal", "power"]))
    assert np.array_equal(_metrics(env), m), "set_state changed the running metrics"
    for how in ("state", "reference", "synthetic"):
        if how == "state":
            env.reset(synthetic_state(env.props, R, seed=4))
        else:
            env.reset(device_mode=how)
        assert not _metrics(env).any(), f"reset({how}): the running metrics did not start from zero"
        run(2)


def test_sharded_cluster_reset_starts_from_zero():
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    n, R = 3000, 2
    env = ShardedClusterEnv(prop(n), R, rank=0, world=1, noise="philox", seed=9)
    env.reset(seed=3)
    rng = np.random.default_rng(5)
    for _ in range(3):
        env.step(_acts(rng, R, n))
    m = _metrics(env)
    assert np.all(m[:, 0] == 3), m
    env.sim.set_state({"signal": np.full(R, 1.0e6)})
    assert np.array_equal(_metrics(env), m), "set_state changed the running metrics"
    env.reset(seed=4)
    assert not _metrics(env).any(), "ShardedClusterEnv.reset: the running metrics did not start from zero"


# ---- the rollout reduction ---------------------------------------------------------------------------
def test_reduce_rollout_metrics_and_replica_shards():
    """One handle of R replicas, checked step by step, against the restated sums through ``reduce_rollout_metrics``;
    the same replicas split over two handles with ``replica_shard`` (Philox is keyed by the global replica)."""
    import torch

    from marl_demandresponse_b200.distributed import reduce_rollout_metrics, replica_shard

    n, R, T = 37, 9, 6
    rng = np.random.default_rng(6)
    acts = (rng.random((T, R, n)) < 0.5).astype(np.uint8)
    whole = _env(n, R, "f32")
    whole.reset()
    halves = []
    for rank in range(2):
        off, k = replica_shard(R, rank, 2)
        h = _env(n, k, "f32", rep_offset=off)
        h.reset()
        halves.append((off, k, h))
    want, tol = np.zeros((R, 6)), np.zeros((R, 6))
    for t in range(T):
        a = torch.as_tensor(acts[t], device="cuda")
        w, e = _checked(whole, lambda: whole.step(a), f"step {t}")
        want += w
        tol += e
        for off, k, h in halves:
            h.step(a[off:off + k].contiguous())
    got = _metrics(whole)
    check_metric_delta(got, want, tol, "whole handle: sums over the episode", sums=(got, got), n_terms=T)
    for off, k, h in halves:
        check_metric_delta(_metrics(h), got[off:off + k], tol[off:off + k], f"replicas [{off}, {off + k})",
                           sums=(got[off:off + k], got[off:off + k]), n_terms=T)

    s = want.sum(axis=0)
    steps = s[0]
    expect = {"replicas": float(R), "replica_steps": steps, "mean_reward": s[1] / steps, "mean_abs_temp_offset": s[2] / steps,
              "rms_temp_error": (s[3] / steps) ** 0.5, "mean_abs_signal_error": s[4] / steps,
              "rms_signal_error": (s[5] / steps) ** 0.5}
    for m in (whole.metrics, torch.cat([h.metrics for _, _, h in halves])):
        res = reduce_rollout_metrics(m)
        assert set(res) == set(expect), sorted(res)
        assert res["replicas"] == expect["replicas"] and res["replica_steps"] == expect["replica_steps"], res
        for key, v in expect.items():
            assert abs(res[key] - v) <= 1e-5 * (abs(v) + 1.0), (key, res[key], v)


# ---- ReferenceMetrics -------------------------------------------------------------------------------
SHAPES = [(1, 10), (7, 37), (5, 256), (3, 257), (300, 100), (2, 1000), (2, 2500)]


def _ref_inputs(env):
    """Absolute temperatures as ``k_metrics_ref`` rebuilds them (fp32: deviation + set-point in fp64; fp64: (Ta -
    target) + target), set-points and rewards of the real houses, and the cluster power."""
    import torch

    torch.cuda.synchronize()
    v = env.state
    f64 = lambda t: t.double().cpu().numpy()   # noqa: E731
    target = f64(v["target"])
    dev = f64(v["dt_air"]) if v["temp_is_deviation"] else f64(v["t_air"]) - target
    return dev + target, target, f64(v["reward"]), f64(v["power"])


def _check_ref(got, bm, what):
    from oracle.metrics_ref import FIELDS

    want = bm.values
    scale = np.abs(want)
    for signed, absolute in (("cumul_temp_offset", "cumul_temp_error"), ("cumul_signal_offset", "cumul_signal_error")):
        scale[:, FIELDS.index(signed)] = want[:, FIELDS.index(absolute)]
    bad = np.argwhere(~(np.abs(got - want) <= 1e-12 * (1.0 + scale)))
    assert bad.size == 0, (what, [(int(r), FIELDS[f], float(got[r, f]), float(want[r, f])) for r, f in bad[:6]])
    for f in ("max_temp_error", "cumul_squared_max_error_temp"):
        i = FIELDS.index(f)
        assert np.array_equal(got[:, i], want[:, i]), (what, f)


@pytest.mark.parametrize("start", [0, 5])
@pytest.mark.parametrize("R,n", SHAPES)
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_reference_metrics_against_the_batched_restatement(precision, R, n, start):
    from marl_demandresponse_b200.metrics import ReferenceMetrics
    from oracle.metrics_ref import BatchedRefMetrics

    env = _env(n, R, precision)
    _reset_across_target(env)
    rng = np.random.default_rng(7)
    m = ReferenceMetrics(env, start_stats_from=start)
    for t in range(2):             # values for initialize() to clear
        m.begin_step()
        env.step(_acts(rng, R, n))
        m.end_step(t)
    assert m.values()[:, 0].any()
    m.initialize()
    bm = BatchedRefMetrics(R, n, start)
    T = 12
    for t in range(T):
        prev = env.get_state(["signal", "od_temp", "power"])
        m.begin_step()
        _plant_padding(env)
        env.step(_acts(rng, R, n))
        _plant_padding(env)
        m.end_step(t)
        ta, target, rew, power = _ref_inputs(env)
        bm.update(ta, target, rew, prev["signal"], power, prev["od_temp"], prev["power"], t)
        _check_ref(m.values(), bm, f"step {t}")
        if t == 5:
            m.reset()
            bm.reset()
            _check_ref(m.values(), bm, "after reset")
    logged = m.log_values(T)
    v = bm.values / float(T)
    from oracle.metrics_ref import FIELDS

    for key, field in (("Mean train return", "cumul_avg_reward"), ("Mean temperature offset", "cumul_temp_offset"),
                       ("Mean temperature error", "cumul_temp_error"), ("Mean signal error", "cumul_signal_offset"),
                       ("Mean signal offset", "cumul_signal_offset"), ("Mean outside temperature", "cumul_OD_temp"),
                       ("Mean signal", "cumul_signal"), ("Mean consumption", "cumul_cons")):
        w = v[:, FIELDS.index(field)]
        assert np.all(np.abs(logged[key] - w) <= 1e-12 * (1.0 + np.abs(w))), key
    rms, want = m.rms(T), bm.rms(T)
    for key, w in want.items():
        assert np.all(np.abs(rms[key] - w) <= 1e-12 * (1.0 + np.abs(w))), key


def test_reference_metrics_refused_on_a_house_sharded_handle():
    from marl_demandresponse_b200._lib import DrsimError
    from marl_demandresponse_b200.metrics import ReferenceMetrics
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    env = ShardedClusterEnv(prop(4000), 1, rank=0, world=2, noise="philox", seed=9)
    env.reset(seed=3)
    m = ReferenceMetrics(env)
    m.begin_step()
    with pytest.raises(DrsimError, match="house-sharded"):
        m.end_step(0)
