"""The device's interpolated base power against the scipy reference of ``interp_ref``, point by point.

* planted points: R one-house clusters, one point per replica (every node, both ends of every axis, the nearest-cell
  midpoints and ties, hour 0 / 86399, day 1 / 364 / 365 / 366), fired by ``refresh(True)`` and by a step with
  injected outdoor-temperature noise (the new datetime and outdoor temperature reach the interpolator);
* the nearest cell from both writers: ``set_state`` (host) and ``drsim_reset`` (device), the latter against
  ``philox.reset_state``;
* the sampled houses: the Philox draw keyed by (seed, global replica, step count) with ``rep_offset`` != 0, at
  N = k, N = k + 1, k = 1 and N >> k, and injected ``interp_ids`` overriding it;
* the interpolator's counter: a reset fires it whatever the previous episode left, a refresh that does not fire
  advances it like the reference, and ``set_state`` refuses per-replica values.

Tolerances: fp64 1e-12 relative; fp32 the first-principles bound of ``interp_ref.sum_bound``.
"""
import copy

import numpy as np
import pytest

import interp_ref as ir
from oracle.config import normalize_env_prop, synthetic_table

pytestmark = pytest.mark.gpu

TABLE = synthetic_table(7)
DT = 4
PERIOD = 300
WORST = {}   # largest fp32 error / bound seen, reported at the end of the module


def _prop(n, k=100, period=PERIOD, solar=True, sig="flat"):
    return {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": float(DT),
            "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0, "solar_gain": solar}},
            "power_grid_prop": {"base_power_props": {"mode": "interpolation", "interp_update_period": period,
                                                     "interp_nb_agents": k},
                                "signal_properties": {"mode": sig}}}


def _defaults(prop):
    hp = normalize_env_prop(prop)["cluster_prop"]["house_prop"]
    return {"dUa": hp["Ua"], "dCm": hp["Cm"], "dCa": hp["Ca"], "dHm": hp["Hm"]}


def _check(env, prop, thermal, ids_of, what):
    """The device's base power on every replica against ``ref_base_power`` on its own planes; ``ids_of(r)`` = the
    sampled houses of replica r."""
    p = normalize_env_prop(prop)
    N, k = env.n_houses, p["power_grid_prop"]["base_power_props"]["interp_nb_agents"]
    solar = p["cluster_prop"]["house_prop"]["solar_gain"]
    fp32 = env.sim.real != np.float64
    st = env.get_state()
    h = _defaults(prop)
    for r in range(env.n_replicas):
        house = {key: st[key][r] for key in ("t_air", "t_mass", "target", "cap")}
        # (the nearest cell is taken from the fp64 capacity given to set_state, not from the fp32 plane: ``thermal``
        # carries it when it matters, e.g. 12500 W + 1e-6)
        house.update({key: np.broadcast_to(thermal[key], (env.n_replicas, N))[r]
                      for key in ("Ua", "Cm", "Ca", "Hm", "cap") if key in thermal})
        ids = np.arange(N) if N <= k else ids_of(r)
        want, tol = ir.ref_base_power(TABLE, house, h, ids, st["od_temp"][r], st["epoch"][r], solar, N, k, fp32)
        err = abs(st["base_power"][r] - want)
        assert err <= tol, f"{what}: replica {r}: base power {st['base_power'][r]!r} != {want!r} (error {err:.3e} > {tol:.3e})"
        if fp32:
            WORST[what] = max(WORST.get(what, (0.0, 0.0, 0.0)), (err / tol, err, tol))
    return st


def _epoch(hour, day):
    """Naive epoch of ``hour`` seconds into 1-based day ``day`` (366: the last day of the leap year 2020)."""
    import datetime as _dt

    year = 2020 if day == 366 else 2021
    w = _dt.datetime(year, 1, 1) + _dt.timedelta(days=int(day) - 1, seconds=int(hour))
    return int((w - _dt.datetime(1970, 1, 1)).total_seconds())


def _planted(prop, R):
    """One point of ``interp_ref.point_set`` per replica of a one-house cluster: state and thermal parameters."""
    pts = ir.point_set(np.random.default_rng(17), m_random=60)
    M = pts["x"].shape[0]
    sel = np.arange(R) % M
    x, ratios, cap = pts["x"][sel], pts["ratios"][:, sel], pts["cap"][sel]
    rng = np.random.default_rng(18)
    h = _defaults(prop)
    target = 19.0 + np.abs(rng.normal(0, 1, R))
    hour = np.clip(np.round(x[:, 3]), 0, 86399)
    day = np.clip(np.round(x[:, 4]), 1, 366)
    thermal = {"Ua": (ratios[0] * h["dUa"])[:, None], "Cm": (ratios[1] * h["dCm"])[:, None],
               "Ca": (ratios[2] * h["dCa"])[:, None], "Hm": (ratios[3] * h["dHm"])[:, None], "cap": cap[:, None]}
    st = {"t_air": (target + x[:, 0])[:, None], "t_mass": (target + x[:, 1])[:, None], "target": target[:, None],
          "on": np.zeros((R, 1), bool), "lockout": np.zeros((R, 1), bool),
          "sso": np.full((R, 1), 100, np.int32), "epoch": np.array([_epoch(a, b) for a, b in zip(hour, day)], np.int64),
          "od_temp": target + x[:, 2], "signal": np.zeros(R), "base_power": np.zeros(R), "power": np.zeros(R),
          "t_since_interp": np.full(R, PERIOD + 1, np.int32), **thermal}
    return st, thermal


@pytest.mark.parametrize("solar", [True, False])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_planted_points_refresh(precision, solar):
    from marl_demandresponse_b200 import BatchedEnv

    prop = _prop(1, solar=solar)
    R = 400
    st, thermal = _planted(prop, R)
    env = BatchedEnv(prop, R, precision=precision, obs_layout="none", seed=3, interp_table=TABLE)
    env.set_state(st)
    env.sim.refresh(True)
    got = _check(env, prop, thermal, None, f"refresh {precision} solar={solar}")
    assert np.all(got["t_since_interp"] == 0)
    assert np.array_equal(got["epoch"], st["epoch"])


@pytest.mark.parametrize("solar", [True, False])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_planted_points_step_with_injected_noise(precision, solar):
    """The interpolator inside a step: the new datetime (epoch + dt) and the new outdoor temperature (the injected
    noise planted so that it lands on the point), the post-update temperatures."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from oracle.np_oracle import from_epoch, od_temp_scalar

    prop = _prop(1, solar=solar)
    p = normalize_env_prop(prop)
    R = 400
    st, thermal = _planted(prop, R)
    st["epoch"] = st["epoch"] - DT
    od_want = st["od_temp"].copy()
    noise = np.array([o - od_temp_scalar(from_epoch(e + DT), p["temp_prop"], 0.0) for o, e in zip(od_want, st["epoch"])])
    env = BatchedEnv(prop, R, precision=precision, obs_layout="none", seed=3, interp_table=TABLE)
    env.set_state(st)
    env.step(torch.zeros((R, 1), dtype=torch.uint8, device="cuda"), od_noise=torch.as_tensor(noise, device="cuda"))
    assert env.sim.last_route in ("k_shard", "four-kernel"), env.sim.last_route
    got = _check(env, prop, thermal, None, f"step {precision} solar={solar}")
    assert np.array_equal(got["epoch"], st["epoch"] + DT)
    want_od = [od_temp_scalar(from_epoch(e + DT), p["temp_prop"], n) for e, n in zip(st["epoch"], noise)]
    np.testing.assert_allclose(got["od_temp"], want_od, rtol=1e-12)
    np.testing.assert_allclose(got["od_temp"], od_want, rtol=1e-12)
    assert np.all(got["t_since_interp"] == 0)


@pytest.mark.parametrize("quirk_ua", [True, False])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_device_reset_cells(precision, quirk_ua):
    """``drsim_reset`` writes the nearest cell on the device: the reset's firing against ``philox.reset_state``'s
    thermal parameters."""
    from marl_demandresponse_b200 import BatchedEnv
    from oracle import philox

    prop = _prop(3)
    R, seed, off = 300, 41, 5
    env = BatchedEnv(prop, R, precision=precision, obs_layout="none", seed=seed, rep_offset=off, interp_table=TABLE)
    env.reset(device_mode="synthetic", quirk_ua=quirk_ua)
    ref = philox.reset_state(seed, R, prop, mode="synthetic", quirk_ua=quirk_ua, rep_offset=off)
    thermal = {k: ref[k] for k in ("Ua", "Cm", "Ca", "Hm")}
    assert np.array_equal(env.get_state(["cap"])["cap"], ref["cap"])
    _check(env, prop, thermal, None, f"drsim_reset {precision} quirk_ua={quirk_ua}")


ID_CASES = [(100, 100), (101, 100), (37, 1), (3000, 10)]


@pytest.mark.parametrize("n,k", ID_CASES)
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_sampled_ids(precision, n, k):
    """The sampled houses: Philox ids of (seed, rep_offset + r, step count) at the reset's firing, a refresh after two
    steps (``set_state`` keeps the step count) and a firing step; injected ``interp_ids`` override the draw."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle import philox

    prop = _prop(n, k=k, sig="sinusoidals")
    R, seed, off = 48, 29, 1000
    st = synthetic_state(prop, R, seed=8, rep_offset=off)
    thermal = {key: st[key] for key in ("Ua", "Cm", "Ca", "Hm")}
    env = BatchedEnv(prop, R, precision=precision, obs_layout="none", seed=seed, rep_offset=off, interp_table=TABLE)
    env.reset(copy.deepcopy(st))
    philox_ids = lambda step: (lambda r: philox.interp_choices(seed, off + r, step, k, n))  # noqa: E731
    _check(env, prop, thermal, philox_ids(0), f"ids {precision} N={n} k={k} reset")
    zeros = torch.zeros((R, n), dtype=torch.uint8, device="cuda")
    for _ in range(2):
        env.step(zeros)
    assert env.get_state(["t_since_interp"])["t_since_interp"].tolist() == [2 * DT] * R
    assert env.sim.step_count == 2
    env.set_state({"t_since_interp": np.full(R, PERIOD + 1, np.int32)})
    env.sim.refresh(True)
    st2 = _check(env, prop, thermal, philox_ids(2), f"ids {precision} N={n} k={k} refresh")
    if n > k:   # a draw keyed by another step or replica would have been caught
        caught = 0
        for r in range(R):
            house = {key: st2[key][r] for key in ("t_air", "t_mass", "target", "cap")}
            house.update({key: thermal[key][r] for key in thermal})
            args = (house, _defaults(prop))
            rest = (st2["od_temp"][r], st2["epoch"][r], True, n, k, precision == "f32")
            want, tol = ir.ref_base_power(TABLE, *args, philox_ids(2)(r), *rest)
            other, _ = ir.ref_base_power(TABLE, *args, philox_ids(3)(r), *rest)
            caught += abs(other - want) > 100 * tol
        assert caught >= 0.9 * R, caught
    # injected ids on a firing step
    inj = np.random.default_rng(4).integers(0, n, (R, k)).astype(np.int32)
    env.set_state({"t_since_interp": np.full(R, PERIOD + 1, np.int32)})
    env.step(zeros, interp_ids=torch.as_tensor(inj, device="cuda"))
    _check(env, prop, thermal, lambda r: inj[r], f"ids {precision} N={n} k={k} injected")
    # a firing step on the draw: keyed by the step count before the step
    env.set_state({"t_since_interp": np.full(R, PERIOD + 1, np.int32)})
    assert env.sim.step_count == 3
    env.step(zeros)
    _check(env, prop, thermal, philox_ids(3), f"ids {precision} N={n} k={k} step")


# ---- the interpolator's counter -----------------------------------------------------------------
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_second_reset_fires_the_interpolator(precision):
    """Two episodes on one handle: the second ``reset(state)``, a few steps into the first, fires the interpolator
    as the reference's new ``PowerGrid`` does, whatever counter the first episode left."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.np_oracle import NpOracle, from_epoch

    prop = _prop(20, sig="sinusoidals")
    R = 16
    env = BatchedEnv(prop, R, precision=precision, obs_layout="none", seed=6, interp_table=TABLE)
    env.reset(synthetic_state(prop, R, seed=1))
    for _ in range(3):
        env.step(torch.zeros((R, 20), dtype=torch.uint8, device="cuda"))
    st = synthetic_state(prop, R, seed=2)
    env.reset(copy.deepcopy(st))
    thermal = {key: st[key] for key in ("Ua", "Cm", "Ca", "Hm")}
    got = _check(env, prop, thermal, None, f"second reset {precision}")
    assert np.all(got["t_since_interp"] == 0), got["t_since_interp"]
    # the signal of the reset's power-grid step, on the device's base power
    orc = NpOracle(prop, R, table=TABLE)
    orc.set_state({**got, **thermal, "t_since_interp": np.full(R, PERIOD + 1)})
    orc.interpolate_power = lambda r, when, ids: got["base_power"][r]
    orc.power_grid_step([from_epoch(e) for e in got["epoch"]])
    np.testing.assert_allclose(got["signal"], orc.state["signal"], rtol=1e-12)
    assert np.all(got["signal"] > 0)


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_refresh_without_firing_advances_the_counter(precision):
    """A reset with ``t_since_interp = 0`` and period 12: the reset's power-grid step adds dt without firing, on the
    device as in the oracle; a ``set_state(get_state())`` round trip then fires on the same step as the handle that
    was not interrupted."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.np_oracle import NpOracle, from_epoch
    from oracle_driver import same_state

    prop = _prop(20, period=12, sig="sinusoidals")
    R = 8
    env = BatchedEnv(prop, R, precision=precision, obs_layout="none", seed=6, interp_table=TABLE)
    st = synthetic_state(prop, R, seed=1)
    st["t_since_interp"] = np.zeros(R, np.int32)
    st["base_power"] = np.full(R, 1234.5)
    env.reset(copy.deepcopy(st))
    orc = NpOracle(prop, R, table=TABLE)
    orc.set_state(st)
    orc.power_grid_step([from_epoch(e) for e in orc.state["epoch"]])
    got = env.get_state()
    assert got["t_since_interp"].tolist() == orc.state["t_since_interp"].tolist() == [DT] * R
    assert np.all(got["base_power"] == 1234.5)
    twin = env.clone()
    env.set_state(env.get_state())
    fired = []
    rng = np.random.default_rng(0)
    for t in range(4):
        a = torch.as_tensor((rng.random((R, 20)) < 0.5).astype(np.uint8), device="cuda")
        env.step(a)
        twin.step(a)
        torch.cuda.synchronize()
        tsi = env.get_state(["t_since_interp"])["t_since_interp"]
        assert np.array_equal(tsi, twin.get_state(["t_since_interp"])["t_since_interp"]), t
        same_state(env, twin)
        if tsi[0] == 0:
            fired.append(t)
    assert fired == [1], fired


def test_set_state_refuses_per_replica_counters():
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200._lib import DrsimError

    prop = _prop(4)
    env = BatchedEnv(prop, 3, obs_layout="none", seed=6, interp_table=TABLE)
    env.reset()
    before = env.get_state(["t_since_interp"])["t_since_interp"].copy()
    with pytest.raises(DrsimError, match="t_since_interp"):
        env.set_state({"t_since_interp": np.array([0, 4, 8], np.int32)})
    assert np.array_equal(env.get_state(["t_since_interp"])["t_since_interp"], before)
    env.set_state({"t_since_interp": np.array([8, 8, 8], np.int32)})
    assert env.get_state(["t_since_interp"])["t_since_interp"].tolist() == [8, 8, 8]


# ---- the other ways in --------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_house_sharded_interpolation_matches_oracle(precision):
    """One 3000-house cluster over three house-sharded handles on one GPU (the partials gathered by hand): each shard
    adds the sampled houses it owns.  ``ShardedClusterEnv.reset`` starts a new episode, so the first step fires; the
    base power is checked against the reference on the whole cluster's planes, and each step re-anchored on the
    oracle of the whole cluster."""
    import torch

    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.sharded import ShardedClusterEnv
    from oracle import philox
    from oracle.np_oracle import NpOracle
    from oracle_driver import od_noise

    n, k, R, W, T, seed = 3000, 100, 2, 3, 8, 9
    prop = _prop(n, k=k, period=12, sig="sinusoidals")
    st = synthetic_state(prop, R, seed=3)
    thermal = {key: st[key] for key in ("Ua", "Cm", "Ca", "Hm")}
    parts = [ShardedClusterEnv(prop, R, rank=r, world=W, precision=precision, obs_layout="tarmac", seed=seed)
             for r in range(W)]
    for p_ in parts:
        p_.sim.set_interp_table(TABLE)
        p_.reset(copy.deepcopy(st))
    h = _defaults(prop)
    acts = (np.random.default_rng(2).random((T, R, n)) < 0.5).astype(np.uint8)
    fired = []
    for t in range(T):
        pre = [p_.sim.get_state() for p_ in parts]
        whole = {key: np.concatenate([s[key] for s in pre], axis=1) for key in ("t_air", "t_mass", "target", "cap", "on",
                                                                                   "lockout", "sso")}
        whole.update({key: pre[0][key] for key in ("epoch", "od_temp", "signal", "base_power", "power", "solar",
                                                   "artificial_ratio", "max_power", "t_since_interp")})
        a = torch.as_tensor(acts[t], device="cuda")
        for p_ in parts:
            p_.sim.views()["actions"].copy_(a[:, p_.lo:p_.hi])
            p_.sim.step_begin(None)
        gathered = torch.stack([p_.state["acc"] for p_ in parts]).contiguous()
        for p_ in parts:
            p_.sim.step_finish(gathered, W)
        torch.cuda.synchronize()
        post = [p_.sim.get_state() for p_ in parts]
        for s in post[1:]:
            for key in ("base_power", "signal", "t_since_interp", "epoch"):
                assert np.array_equal(s[key], post[0][key]), (t, key)
        got = {key: np.concatenate([s[key] for s in post], axis=1) for key in ("t_air", "t_mass", "target", "cap")}
        got.update({key: post[0][key] for key in ("epoch", "od_temp", "signal", "base_power", "power", "t_since_interp")})
        ids = [philox.interp_choices(seed, r, t, k, n) for r in range(R)]
        if got["t_since_interp"][0] == 0:
            fired.append(t)
            owners = {j for i in ids[0] for j, p_ in enumerate(parts) if p_.lo <= i < p_.hi}
            assert owners == set(range(W)), owners   # every shard adds some of the sampled houses
            for r in range(R):
                house = {key: got[key][r] for key in ("t_air", "t_mass", "target", "cap")}
                house.update({key: thermal[key][r] for key in thermal})
                want, tol = ir.ref_base_power(TABLE, house, h, ids[r], got["od_temp"][r], got["epoch"][r], True, n, k,
                                              precision == "f32")
                assert abs(got["base_power"][r] - want) <= tol, (t, r, got["base_power"][r], want, tol)
        orc = NpOracle(prop, R, table=TABLE)
        orc.set_state({**whole, **thermal})
        orc.interpolate_power = lambda r, when, ids_r: got["base_power"][r]
        orc.step(acts[t], od_noise(seed, range(R), [t])[0], None, np.stack(ids))
        s = orc.state
        assert np.array_equal(got["t_since_interp"], s["t_since_interp"]), t
        np.testing.assert_allclose(got["od_temp"], s["od_temp"], rtol=1e-9)
        np.testing.assert_allclose(got["signal"], s["signal"], rtol=1e-9)
        np.testing.assert_allclose(got["power"], s["power"], rtol=1e-6)
    assert fired == [0, 3, 6], fired


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_host_buffer_steps_across_a_firing_step(precision):
    """``step_host``, ``step_host_full`` and ``step_host_snapshot`` through firing and non-firing steps: the same bits
    as ``step``."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle_driver import same_state

    prop = _prop(300, k=50, period=12, sig="sinusoidals")
    R = 6
    ref = BatchedEnv(prop, R, precision=precision, obs_layout="hand_engineered", seed=12, interp_table=TABLE)
    ref.reset(synthetic_state(prop, R, seed=5))
    others = [ref.clone() for _ in range(3)]
    real = np.float64 if precision == "f64" else np.float32
    rng = np.random.default_rng(1)
    fired = []
    for t in range(7):
        a = (rng.random((R, 300)) < 0.5).astype(np.uint8)
        ref.step(torch.as_tensor(a, device="cuda"))
        others[0].step_host(a)
        others[1].step_host(a, reward_out=np.zeros((R, 300), real), obs_out=np.zeros((R, 300, ref.sim.D), real))
        others[2].sim.step_host_snapshot(a)
        torch.cuda.synchronize()
        for o in others:
            same_state(ref, o)
            assert np.array_equal(o.get_state(["t_since_interp"])["t_since_interp"],
                                  ref.get_state(["t_since_interp"])["t_since_interp"])
        if ref.get_state(["t_since_interp"])["t_since_interp"][0] == 0:
            fired.append(t)
    assert fired == [2, 5], fired


def test_run_matches_the_free_running_oracle():
    """``run(T)`` on an interpolation handle (one launch per step: the in-kernel loop takes the constant base power
    only) against the free-running oracle, fp64; and fp32 ``run(T)`` bit for bit against ``T`` checked steps."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle_driver import OracleDriver, config, same_state

    for precision in ("f64", "f32"):
        p = config(100, sig="regular_steps", **{"power_grid_prop/base_power_props/mode": "interpolation",
                                                 "power_grid_prop/base_power_props/interp_update_period": 10,
                                                 "power_grid_prop/base_power_props/interp_nb_agents": 30})
        R, T = 5, 20
        env = BatchedEnv(p, R, precision=precision, obs_layout="hand_engineered", seed=31, interp_table=TABLE)
        st = synthetic_state(p, R, seed=4)
        env.reset(copy.deepcopy(st))
        tape = (torch.rand((T, R, 100), device="cuda", generator=torch.Generator(device="cuda").manual_seed(6)) < 0.5)
        tape = tape.to(torch.uint8)
        if precision == "f64":
            drv = OracleDriver(env, p, st, table=TABLE)
            drv.start_free()
            env.run(T, tape)
            for t in range(T):
                drv.advance_free(tape[t].cpu().numpy())
            drv.check_free("run(20), interpolated base power")
        else:
            twin = env.clone()
            drv = OracleDriver(twin, p, st, table=TABLE)
            env.run(T, tape)
            for t in range(T):
                drv.step(tape[t].cpu().numpy())
            torch.cuda.synchronize()
            same_state(env, twin)
            assert drv.fired == [t for t in range(T) if t % 3 == 2], drv.fired


def test_report_worst_fp32_error():
    """(Runs last in this module.)  The largest fp32 base-power error seen, next to its bound."""
    for what, (ratio, err, tol) in sorted(WORST.items(), key=lambda kv: -kv[1][0]):
        print(f"fp32 base power, {what}: error / bound {ratio:.3e} (error {err:.3e} W, bound {tol:.3e} W)")
