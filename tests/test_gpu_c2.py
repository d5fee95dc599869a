"""BASELINE config 2 as a whole, against the oracle: ONE 1,000-house cluster, base power interpolated in the
Monte-Carlo table (power_grid.py:130-161, interpolation.py:137-243) -- the table GENERATED on the GPU by the
restated v0/monteCarlo/monteCarlo.py:152-230, the reference's own .npy being absent from the checkout --, 100
houses re-sampled on every update, lock-out 40 s, greedy-myopic controller in closed loop
(greedy_myopic_controller.py:67-104), perlin-type signal and outdoor-temperature noise from the device's
Philox streams.  170 steps: the interpolator fires at reset, after 75 and after 150 steps.
"""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, R, T, SEED = 1000, 1, 170, 4242

_TABLE = {}


def _table():
    if "t" not in _TABLE:
        from marl_demandresponse_b200.montecarlo import generate_table

        _TABLE["t"] = generate_table()   # all 4,199,040 entries, a few seconds on the GPU
    return _TABLE["t"]


def _prop():
    return {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
            "cluster_prop": {"nb_agents": N, "house_prop": {"target_temp": 19.0, "hvac_prop": {"lockout_duration": 40}}},
            "power_grid_prop": {"base_power_props": {"mode": "interpolation", "interp_update_period": 300, "interp_nb_agents": 100},
                                "signal_properties": {"mode": "perlin"}}}


def _noise(st):
    """What the device's Philox streams must produce: outdoor-temperature draws, signal noise, sampled house ids."""
    from oracle import philox

    epoch0 = int(st["epoch"][0])
    od = np.array([[philox.od_noise(SEED, 0, t, 1.0)] for t in range(T)])
    per = np.array([[philox.perlin(SEED, 0, ((epoch0 + 4 * t) % 86400) / 300.0, 5, 5)] for t in range(T + 1)])
    ids = {t: philox.interp_choices(SEED, 0, t, 100, N)[None] for t in range(T)}
    return od, per, ids


def test_generated_table_is_a_table():
    t = _table()
    assert t.shape == (4_199_040,) and np.isfinite(t).all()
    # average bang-bang power of a 10 / 15 kW unit with cop 2.5: between 0 and capacity / cop
    assert t.min() >= 0.0 and t.max() <= 15000.0 / 2.5 + 1e-6 and t.std() > 100.0


def test_c2_closed_loop_fp64_matches_oracle():
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.np_oracle import NpOracle, from_epoch, greedy_myopic

    prop, table = _prop(), _table()
    st = synthetic_state(prop, R, seed=21)
    od, per, ids = _noise(st)
    env = BatchedEnv(prop, R, precision="f64", policy="greedy_myopic", noise="philox", seed=SEED, interp_table=table)
    env.reset(copy.deepcopy(st))
    orc = NpOracle(prop, R, table=table)
    orc.set_state(copy.deepcopy(st))
    orc.power_grid_step([from_epoch(e) for e in orc.state["epoch"]], per[0], ids[0])   # PowerGrid.step at reset: first firing
    fired, base_seen, rewards = [], set(), []
    for t in range(T):
        s = orc.state
        a = np.stack([greedy_myopic(s["t_air"][r], s["target"][r], s["cap"][r], 2.5, s["lockout"][r], s["signal"][r]) for r in range(R)])
        tsi = int(s["t_since_interp"][0])
        rew = orc.step(a, od[t], per[t + 1], ids[t])
        if int(orc.state["t_since_interp"][0]) < tsi:
            fired.append(t)
        base_seen.add(float(orc.state["base_power"][0]))
        env.step(None)
        rewards.append(rew)
    assert fired == [74, 149], fired           # the interpolator fired twice after the reset
    assert len(base_seen) >= 3                 # ... and moved the base power each time
    got = env.get_state()
    s = orc.state
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k].astype(np.int64), s[k].astype(np.int64)), k
    assert np.array_equal(got["epoch"], s["epoch"])
    np.testing.assert_allclose(got["t_air"], s["t_air"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(got["t_mass"], s["t_mass"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(got["base_power"], s["base_power"], rtol=1e-11)
    np.testing.assert_allclose(got["signal"], s["signal"], rtol=1e-11)
    np.testing.assert_allclose(got["power"], s["power"], rtol=1e-12)
    np.testing.assert_allclose(env.reward.double().cpu().numpy(), rewards[-1], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(env.obs.double().cpu().numpy(), orc.obs_vectors(), rtol=1e-9, atol=1e-9)


def test_c2_fp32_on_the_oracle_action_tape():
    """The production fp32 build on the same configuration, driven by the oracle's greedy-myopic actions (an
    fp32 temperature within an ulp of another house's would reorder the greedy scan: SURVEY 7.3-1): discrete
    state bit-exact, continuous state within the fp32 tolerance."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.np_oracle import NpOracle, from_epoch, greedy_myopic

    prop, table = _prop(), _table()
    st = synthetic_state(prop, R, seed=21)
    od, per, ids = _noise(st)
    env = BatchedEnv(prop, R, precision="f32", policy="external", noise="philox", seed=SEED, interp_table=table)
    env.reset(copy.deepcopy(st))
    orc = NpOracle(prop, R, table=table)
    orc.set_state(copy.deepcopy(st))
    orc.power_grid_step([from_epoch(e) for e in orc.state["epoch"]], per[0], ids[0])
    for t in range(T):
        s = orc.state
        a = np.stack([greedy_myopic(s["t_air"][r], s["target"][r], s["cap"][r], 2.5, s["lockout"][r], s["signal"][r]) for r in range(R)])
        rew = orc.step(a, od[t], per[t + 1], ids[t])
        env.step(torch.as_tensor(a.astype(np.uint8), device="cuda"))
    got = env.get_state()
    s = orc.state
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k].astype(np.int64), s[k].astype(np.int64)), k
    np.testing.assert_allclose(got["t_air"], s["t_air"], rtol=0, atol=1e-5 * 40)
    np.testing.assert_allclose(got["base_power"], s["base_power"], rtol=1e-5)
    np.testing.assert_allclose(got["signal"], s["signal"], rtol=1e-5)
    np.testing.assert_allclose(got["power"], s["power"], rtol=1e-6)
    np.testing.assert_allclose(env.reward.double().cpu().numpy(), rew, rtol=1e-5, atol=1e-5 * 2)
    np.testing.assert_allclose(env.obs.double().cpu().numpy(), orc.obs_vectors(), rtol=1e-5, atol=1e-5)


def test_c2_fp32_greedy_on_the_device():
    """The production fp32 build with greedy-myopic on the device, as benchmarked.  Every step the action plane
    ``k_greedy`` wrote is the restated greedy on the device's own inputs (fp32 deviation from the set-point as the key,
    capacities, lock-out bits, the signal before the step), and the discrete state is those actions through the lock-out
    state machine.  The continuous state under these actions is ``test_c2_fp32_on_the_oracle_action_tape``'s."""
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.np_oracle import hvac_fsm
    from oracle_driver import check_greedy_plane, controller_actions, controller_inputs

    prop, table = _prop(), _table()
    st = synthetic_state(prop, R, seed=21)
    env = BatchedEnv(prop, R, precision="f32", policy="greedy_myopic", noise="philox", seed=SEED, interp_table=table)
    env.reset(copy.deepcopy(st))
    s = env.get_state(["on", "lockout", "sso"])
    on, lock, sso = s["on"], s["lockout"], s["sso"]
    n_on = []
    for t in range(T):
        want = controller_actions("greedy_myopic", 0.0, 2.5, **controller_inputs(env))
        env.step(None)
        check_greedy_plane(env, want, f"step {t}")
        on, lock, sso = hvac_fsm(on, lock, sso, want, 4, 40)
        got = env.get_state(["on", "lockout", "sso"])
        for k, v in (("on", on), ("lockout", lock), ("sso", sso)):
            assert np.array_equal(got[k].astype(np.int64), v.astype(np.int64)), (t, k)
        n_on.append(int(want.sum()))
    assert 0 < min(n_on) and max(n_on) < N, (min(n_on), max(n_on))   # the signal splits the cluster every step
