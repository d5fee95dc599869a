"""The on-device controllers against the reference controllers of ``oracle.np_oracle``, on every step route.

The controllers are written out in several kernels: deadband bang-bang, bang-bang and always-on in
``house4_step_f32`` (``k_fused_direct``), ``house4_compute_f32`` (``k_fused_tma<0>``, ``k_shard``), ``policy_action``
(``k_house``, chunked ``k_fused``, the fp64 kernels), ``k_small`` and the first phase of ``k_shard``; greedy-myopic in
``k_greedy`` ahead of the step kernel.  The reference controllers are fed the device's own pre-step planes
(``oracle_driver.controller_inputs``), so every action must match exactly:

* greedy-myopic writes the action plane: it must equal the reference on every house of every replica, and the
  padding slots must be 0;
* the bang-bang family writes no action plane: its actions are checked through the lock-out state machine, the
  reference actions advanced by ``hvac_fsm`` against the device's ``on`` / ``lockout`` / ``sso`` bit for bit.

Cases: one step from planted states at the thresholds and edges (``test_bangbang_family_at_the_thresholds``, the greedy
shape and value cases), 24 steps in closed loop on every route (``test_closed_loop_matches_reference_controller``),
the in-kernel step loop under a controller (``test_in_kernel_loop_under_controller``), and the limits of greedy-myopic.
"""
import copy
import zlib

import numpy as np
import pytest

from oracle_driver import (ROUTES, OracleDriver, check_greedy_plane, config, controller_actions, controller_inputs,
                           loop_launches, prop, same_state)

pytestmark = pytest.mark.gpu

T_STEPS = 24

# routes that are not cells of the external-action route matrix: k_shard on plain rows (TarMAC, 10 columns: its early
# cluster-power pre-pass restates the controllers) and the four-kernel path of the fp64 build
EXTRA_ROUTES = {
    "k_shard/plain": ("f32", 2, 2500, "tarmac", "auto", {}, dict(route="k_shard", variant="none", launches=1)),
    "four-kernel<double>": ("f64", 24, 100, "hand_engineered", "split", {"DRSIM_NO_SHARD_KERNEL": 1},
                            dict(route="four-kernel", variant="none", launches=4)),
}
POLICIES = ("deadband_bangbang", "bangbang", "always_on", "greedy_myopic")
BANGBANG_FAMILY = POLICIES[:3]
F32_ROUTES = ("k_small", "k_fused_tma<0>/1-per-tile", "k_fused_tma<0>/3-per-tile", "k_fused_rows<staged>",
              "k_fused_rows<unstaged>", "k_fused/chunked", "k_fused_direct", "k_shard", "k_shard/plain", "four-kernel")
F64_ROUTES = ("k_small_gen<double>", "k_fused_direct<double>", "k_fused<double>/chunked", "k_shard<double>",
              "four-kernel<double>")


def _route(route):
    return EXTRA_ROUTES[route] if route in EXTRA_ROUTES else ROUTES[route]


# the cell of each route here, from its cells in the external-action matrix: rows that keep the planned tile variant
# and clusters per tile (chunked k_fused: a solar column, or the plain rows would take k_fused_rows)
ROUTE_CELL = {"k_fused_tma<0>/1-per-tile": dict(c=1), "k_fused_tma<0>/3-per-tile": dict(c=2),
              "k_fused_direct": dict(c=1), "k_small": dict(c=9), "four-kernel": dict(c=1),
              "k_small_gen<double>": dict(c=9), "k_fused/chunked": dict(state="solar")}


def _expected(route, policy):
    """(last_route, launches per step) of ``route`` under ``policy``: ``k_fused_rows`` takes its actions from the action
    plane (external or greedy-myopic), the bang-bang family falls back to the four-kernel path there; greedy-myopic
    adds the ``k_greedy`` launch."""
    expect = _route(route)[-1]
    r, n = expect["route"], expect["launches"]
    if route.startswith("k_fused_rows") and policy != "greedy_myopic":
        r, n = "four-kernel", 4
    return r, n + (policy == "greedy_myopic")


def _env(route, policy, monkeypatch, deadband, seed=21, **over):
    """The handle of ``route`` under ``policy`` (reset to the seeded synthetic state), its properties and that state."""
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    precision, R, N, layout, path, env_vars, expect = _route(route)
    for k, v in env_vars.items():
        monkeypatch.setenv(k, str(v))
    over = {**ROUTE_CELL.get(route, {}), **over}
    p = config(N, **{"cluster_prop/house_prop/deadband": deadband}, **over)
    env = BatchedEnv(p, R, precision=precision, obs_layout=layout, policy=policy, noise="philox", seed=seed, path=path)
    info = env.sim.fused_info()
    if "variant" in expect:
        assert info["variant"] == expect["variant"], (route, info)
    if "e" in expect:
        assert info["envs_per_tile"] == expect["e"], (route, info)
    st = synthetic_state(p, R, seed=seed + 1)
    env.reset(copy.deepcopy(st))
    return env, p, st


def _cuda(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


# ---- a) one step from planted states ---------------------------------------------------------------------------
def _threshold_temperatures(env, deadband):
    """Temperatures on the controllers' thresholds: ``±deadband / 2`` and the set-point itself, with their ``nextafter``
    neighbours.  fp32: deviations (``+0.0`` and ``-0.0`` included); fp64: absolute temperatures around each house's
    set-point, the thresholds computed as the reference computes them (``target ± deadband / 2``)."""
    if env.state["temp_is_deviation"]:
        h = np.float32(deadband / 2)
        assert float(h) == deadband / 2, "the fp32 threshold cases need a deadband whose half is exact in fp32"
        edges = [h, -h, np.float32(0.0)]
        devs = [np.float32(-0.0)] + [v for e in edges for v in (e, np.nextafter(e, np.float32(np.inf)),
                                                                 np.nextafter(e, np.float32(-np.inf)))]
        return np.array(devs, dtype=np.float32)
    tgt = env.state["target"].double().cpu().numpy()
    edges = [tgt - deadband / 2, tgt + deadband / 2, tgt]
    return np.stack([v for e in edges for v in (e, np.nextafter(e, np.inf), np.nextafter(e, -np.inf))])   # [K, R, N]


def _plant_bangbang(env, deadband, dur, dt, rng):
    """Every threshold temperature crossed with the three lock-out states (on; off and locked; off and free), spread over
    the batch in a seeded shuffle.  Writes the zero-copy planes."""
    R, N = env.n_replicas, env.n_houses
    temps = _threshold_temperatures(env, deadband)
    # (on, lockout, sso): locked houses one and two steps short of their duration, free ones at and past it
    states = [(1, 0, 0), (0, 1, dur - dt), (0, 1, dur - 2 * dt), (0, 0, dur), (0, 0, dur + dt)]
    n_combo = len(temps) * len(states)
    assert R * N >= n_combo, (R, N, n_combo)
    combo = (rng.permutation(R * N) % n_combo).reshape(R, N)
    ti, si = combo // len(states), combo % len(states)
    s = np.array(states)[si]
    on, lock, sso = s[..., 0], s[..., 1], s[..., 2]
    if temps.ndim == 1:
        env.state["dt_air"].copy_(_cuda(temps[ti]))
    else:
        env.state["t_air"].copy_(_cuda(np.take_along_axis(temps, ti[None], 0)[0]))
    env.state["flags"].copy_(_cuda((on | (lock << 1)).astype(np.uint8)))
    env.state["sso"].copy_(_cuda(sso.astype(np.int32)))


BB_CASES = [(r, pol, 0.5) for r in F32_ROUTES if not r.startswith("k_fused_rows") for pol in BANGBANG_FAMILY]
BB_CASES += [("k_small", "deadband_bangbang", 1.0), ("k_fused_tma<0>/3-per-tile", "deadband_bangbang", 1.0)]
BB_CASES += [(r, pol, 0.4) for r in F64_ROUTES for pol in BANGBANG_FAMILY]


@pytest.mark.parametrize("route,policy,deadband", [pytest.param(*c, id=f"{c[0]}-{c[1]}-{c[2]}") for c in BB_CASES])
def test_bangbang_family_at_the_thresholds(route, policy, deadband, monkeypatch):
    """One step from temperatures exactly on, and one ulp either side of, every threshold, crossed with on / off and
    locked / free houses: the device's discrete state after the step is the reference action through ``hvac_fsm``."""
    env, p, st = _env(route, policy, monkeypatch, deadband)
    drv = OracleDriver(env, p, st)
    _plant_bangbang(env, deadband, drv.dur, int(drv.p["time_step"]), np.random.default_rng(7))
    drv = OracleDriver(env, p, st)      # anchored on the planted discrete state
    inputs = controller_inputs(env)
    want = controller_actions(policy, deadband, drv.cop, **inputs)
    if policy == "deadband_bangbang":   # the planted batch reaches all three verdicts of the dead band, on and off
        hold = ~((inputs["x"] < inputs["target"] - deadband / 2) | (inputs["x"] > inputs["target"] + deadband / 2))
        assert hold.any() and (want & ~hold).any() and (~want & ~hold).any()
    drv.step()
    assert env.sim.last_route == _expected(route, policy)[0], (route, policy, env.sim.last_route)


GREEDY_N = (1, 2, 31, 32, 33, 100, 1000, 1023, 1024, 1025, 2048, 3000, 8192)


def _greedy_env(N, R, precision="f32", cop=2.5):
    from marl_demandresponse_b200 import BatchedEnv

    p = prop(N, **{"cluster_prop/house_prop/hvac_prop/cop": cop})
    env = BatchedEnv(p, R, precision=precision, obs_layout="none", policy="greedy_myopic", noise="zero")
    env.reset()
    return env


def _plant_greedy(env, dev, cap, lock, signal):
    """Deviations from the set-point (fp32 values: the same keys in both builds), capacities, lock-out bits and signals
    on the zero-copy planes; the padding slots of the action plane pre-filled with 1 (``k_greedy`` must clear them)."""
    import torch

    v = env.state
    if v["temp_is_deviation"]:
        v["dt_air"].copy_(_cuda(dev.astype(np.float32)))
    else:   # 19 + dev is exact in fp64, and so is the key (19 + dev) - 19
        v["target"].fill_(19.0)
        v["t_air"].copy_(_cuda(19.0 + dev))
    v["cap"].copy_(_cuda(cap.astype(np.float32 if v["temp_is_deviation"] else np.float64)))
    v["flags"].copy_(_cuda((lock.astype(np.uint8) << 1)))
    v["signal"].copy_(_cuda(np.asarray(signal, dtype=np.float64)))
    v["actions_padded"][:, env.n_houses:] = 1
    torch.cuda.synchronize()


def _greedy_step(env, cop, what):
    want = controller_actions("greedy_myopic", 0.0, cop, **controller_inputs(env))
    env.step(None)
    check_greedy_plane(env, want, what)
    return want


@pytest.mark.parametrize("R", (1, 37, 300))
@pytest.mark.parametrize("N", GREEDY_N)
def test_greedy_shapes(N, R):
    """Both sorts (one element per thread up to 1024 slots, strided in shared memory above), the scan with one and with
    several houses per thread, padded planes (N % 4 != 0), one to 300 replicas."""
    rng = np.random.default_rng(N * 1000 + R)
    env = _greedy_env(N, R)
    dev = rng.uniform(-2.0, 4.0, (R, N)).astype(np.float32).astype(np.float64)
    cap = rng.choice([10000.0, 15000.0], (R, N))
    total = (cap / 2.5).sum(axis=1)
    _plant_greedy(env, dev, cap, rng.random((R, N)) < 0.3, rng.uniform(0.0, 1.1, R) * total)
    want = _greedy_step(env, 2.5, f"N={N} R={R}")
    if N >= 100 and R > 1:   # the signals leave houses on both sides of the verdict
        assert want.any() and not want.all()


def _sorted_order(dev):
    return np.argsort(-dev, axis=1, kind="stable")


def _greedy_values(case, R, N, cop, rng):
    """``(dev, cap, lock, signal, k)`` of one value case (see ``test_greedy_values``); ``k[r]``: the houses whose powers
    sum to the signal in the prefix cases."""
    dev = rng.uniform(-2.0, 4.0, (R, N)).astype(np.float32).astype(np.float64)
    ks = None
    cap = rng.choice([10000.0, 15000.0], (R, N))
    lock = rng.random((R, N)) < 0.3
    if case == "all_equal":
        dev[:] = 0.75
    elif case == "ties":
        # sorted positions in groups of equal keys; two groups straddle position 32 and 1024 (512 below 1050 houses)
        hi = 1024 if N > 1050 else 512
        cuts = [0, 20, 45, hi - 24, hi + 26, N]
        pos_dev = np.concatenate([np.full(b - a, 3.0 - g) for g, (a, b) in enumerate(zip(cuts, cuts[1:]))])
        for r in range(R):
            dev[r, rng.permutation(N)] = pos_dev
    elif case == "zero_cap":
        cap[rng.random((R, N)) < 0.25] = 0.0
    elif case == "mostly_locked":
        lock = rng.random((R, N)) < 0.9
    power = cap / cop
    total = power.sum(axis=1)
    signal = rng.uniform(0.0, 1.1, R) * total
    if case == "signal_nonpositive":
        signal = np.where(np.arange(R) % 2 == 0, 0.0, -rng.uniform(1.0, 1e4, R))
    elif case == "signal_above_total":
        signal = np.where(np.arange(R) % 2 == 0, total, 1.5 * total)
    elif case.startswith("prefix"):
        # the signal equals the running total of the first k houses in greedy order (the reference's own sum): the k-th
        # house reaches it exactly, so the first clause refuses it and the second takes it unless it is locked out
        order = _sorted_order(dev)
        ks = rng.integers(1, N, R)
        for r, k in enumerate(ks):
            t = 0
            for h in order[r, :k]:
                t += power[r, h]
            signal[r] = t
            lock[r, order[r, k - 1]] = case == "prefix_locked"
    return dev, cap, lock, signal, ks


GREEDY_VALUE_CASES = ("random", "all_equal", "ties", "signal_nonpositive", "signal_above_total", "prefix_locked",
                      "prefix_unlocked", "mostly_locked", "zero_cap")


@pytest.mark.parametrize("case", GREEDY_VALUE_CASES)
@pytest.mark.parametrize("precision,N", [("f32", 1000), ("f32", 3000), ("f64", 3000)])
@pytest.mark.parametrize("cop", (2.5, 2.3))
def test_greedy_values(case, precision, N, cop):
    """Keys, signals and powers at the edges of the scan.  cop 2.5 with 10 / 15 kW gives exactly representable powers
    (the parallel-prefix path of ``k_greedy``), cop 2.3 does not (the sequential scan).  Ties are broken by house index
    on the device and in the reference's stable sort."""
    rng = np.random.default_rng(zlib.crc32(f"{case} {precision} {N} {cop}".encode()))
    R = 37
    env = _greedy_env(N, R, precision, cop)
    dev, cap, lock, signal, ks = _greedy_values(case, R, N, cop, rng)
    _plant_greedy(env, dev, cap, lock, signal)
    want = _greedy_step(env, cop, f"{case} {precision} N={N} cop={cop}")
    # what the case is built to reach, in the reference's own verdicts
    if case == "signal_nonpositive":
        assert not want.any()
    if case == "signal_above_total":
        assert want[1::2].all()
    if case.startswith("prefix"):   # the first k - 1 houses taken, the k-th exactly when it is free (then no more)
        order = _sorted_order(dev)
        free = case == "prefix_unlocked"
        for r, k in enumerate(ks):
            w = want[r, order[r]]
            assert w[:k - 1].all() and w[k - 1] == free and not (free and w[k:].any()), (r, k)


def test_greedy_handles_of_different_sizes():
    """Handles of different cluster sizes side by side: a smaller one created after a larger one leaves the larger one
    able to launch its sort."""
    rng = np.random.default_rng(5)
    envs = [(_greedy_env(n, 3), n) for n in (8192, 3000, 100)]
    for env, n in envs[::-1] + envs:
        dev = rng.uniform(-2.0, 4.0, (3, n)).astype(np.float32).astype(np.float64)
        cap = rng.choice([10000.0, 15000.0], (3, n))
        _plant_greedy(env, dev, cap, rng.random((3, n)) < 0.3, 0.5 * (cap / 2.5).sum(axis=1))
        _greedy_step(env, 2.5, f"N={n}")


def test_greedy_cluster_size_limit():
    """8192 houses sort in 192 KB of shared memory; 8193 round up to 16384 slots and are refused at creation."""
    from marl_demandresponse_b200._lib import DrsimError

    _greedy_env(8192, 1)
    with pytest.raises(DrsimError, match="cluster too large for the shared-memory sort"):
        _greedy_env(8193, 1)


def test_house_sharded_greedy_is_refused():
    """Greedy-myopic sorts the whole cluster against its signal: a house-sharded handle refuses it; the bang-bang family
    decides per house and shards."""
    from marl_demandresponse_b200._lib import DrsimError
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    p = prop(64)
    with pytest.raises(DrsimError, match="house-sharded cluster: the greedy scan sorts the whole cluster"):
        ShardedClusterEnv(p, 2, rank=1, world=2, policy="greedy_myopic")
    for policy in BANGBANG_FAMILY:
        for r in range(2):
            ShardedClusterEnv(p, 2, rank=r, world=2, policy=policy)
    ShardedClusterEnv(p, 2, rank=0, world=1, policy="greedy_myopic")   # one rank holds the whole cluster


# ---- b) every route in closed loop ------------------------------------------------------------------------------
LOOP_CASES = [(r, pol) for r in F32_ROUTES + F64_ROUTES for pol in POLICIES]


@pytest.mark.parametrize("route,policy", [pytest.param(*c, id=f"{c[0]}-{c[1]}") for c in LOOP_CASES])
def test_closed_loop_matches_reference_controller(route, policy, monkeypatch):
    """24 steps under the on-device controller, each re-anchored on the oracle stepped with the reference controller's
    actions on the device's pre-step planes; the fp64 build also free-running against the oracle driven by the
    restated controller on its own state.  (An fp32 trajectory drifts from the fp64 oracle by more than an ulp, and a
    free-running controller may then decide differently at a threshold: fp32 is checked re-anchored only.)"""
    f64 = _route(route)[0] == "f64"
    env, p, st = _env(route, policy, monkeypatch, 0.4 if f64 else 0.5, sig="sinusoidals")
    drv = OracleDriver(env, p, st)
    if f64:
        drv.start_free()
    want_route, per_step = _expected(route, policy)
    launches = [drv.step()]
    assert env.sim.last_route == want_route, (route, policy, env.sim.last_route)
    launches += [drv.step() for _ in range(1, T_STEPS)]
    # the first step generates the 64-step schedule block (two kernels)
    assert launches == [per_step + 2] + [per_step] * (T_STEPS - 1), launches
    drv.check_metrics()
    if f64:
        drv.check_free()


# ---- c) the in-kernel step loop under a controller ---------------------------------------------------------------
@pytest.mark.parametrize("policy", BANGBANG_FAMILY)
@pytest.mark.parametrize("route", ("k_small", "k_fused_tma<0>/1-per-tile", "k_fused_tma<0>/3-per-tile"))
def test_in_kernel_loop_under_controller(route, policy, monkeypatch):
    """``run(T)`` with the controller inside the step loop of the kernel (the C1 benchmark's path on ``k_small``): one
    step kernel per schedule block, and the bits of a clone stepped T times through the checked per-step driver."""
    import torch

    T = 70   # crosses the 64-step schedule block
    env, p, st = _env(route, policy, monkeypatch, 0.5)
    twin = env.clone()
    drv = OracleDriver(twin, p, st)
    for _ in range(T):
        drv.step()
    l0 = env.sim.launch_count
    env.run(T)
    torch.cuda.synchronize()
    assert env.sim.last_route == _expected(route, policy)[0], env.sim.last_route
    assert env.sim.launch_count - l0 == loop_launches(0, T, None), env.sim.launch_count - l0
    same_state(env, twin)
