"""Host-side pieces of the drop-in against the reference: neighbour tables for every communication mode
over a sweep of cluster sizes and parameters (same table or the same exception), the per-step
``random_sample`` draw under the same ``random`` seed, the default property tree, the Perlin octave sum,
the interpolation grids, the controllers and the actor architecture.

With the reference checkout present (``DRSIM_REFERENCE_ROOT``) every comparison runs against the RUNNING
reference; without it, against what the reference returns on the same inputs, stored in
``tests/golden/host_vs_reference/`` (``values.json``, ``actor.npz``) (``tests/golden/make_golden_host.py``)."""
import json
import os
import random

import numpy as np
import pytest

from oracle import refenv

LIVE = refenv.available()
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

COMM_MODES = ["neighbours", "closed_groups", "neighbours_2D", "random_fixed"]
SAMPLE_CASES = ((9, 3), (24, 10), (5, 4))
PERLIN_CASES = ((5, 5, 300, 0.37), (3, 2, 120, 0.9), (1, 5, 300, 0.1), (6, 1, 50, 0.5))
PERLIN_X = (0.0, 1.0, 17.5, 299.0, 86399.0)
GREEDY_N = (3, 17, 40, 128)
ACTOR_CASES = ((50, [100, 100]), (10, "[100, 100]"), (46, [64, 48]))


def stored(key):
    with open(os.path.join(GOLDEN, "host_vs_reference", "values.json")) as f:
        return json.load(f)[key]


def _dump(m):
    return m.model_dump() if hasattr(m, "model_dump") else m.dict()


def _props(n, mode, c, dist, row):
    from marl_demandresponse_b200.properties import as_props

    return as_props({"cluster_prop": {"nb_agents": n, "agents_comm_prop": {
        "mode": mode, "max_nb_agents_communication": c, "max_communication_distance": dist, "row_size": row}}})


def comm_cases(mode):
    for n in (2, 3, 4, 5, 9, 10, 12, 16, 20, 25, 36, 40, 100):
        for c in (1, 2, 3, 4, 5, 10, 11):
            for dist, row in ((1, 5), (2, 5), (1, 4), (2, 6), (3, 10)):
                if mode != "neighbours_2D" and (dist, row) != (1, 5):
                    continue
                yield n, c, dist, row


def comm_key(n, c, dist, row):
    return f"{n},{c},{dist},{row}"


def perlin_key(octaves, step, period, seed):
    return f"{octaves},{step},{period},{seed}"


@pytest.mark.parametrize("mode", COMM_MODES)
def test_neighbour_tables_equal_the_reference_builder(mode):
    from marl_demandresponse_b200.environment import build_comm_table

    if LIVE:
        ns = refenv.load()
        Builder = ns.comm_mod.AgentCommunicationBuilder
    else:
        tables = stored("neighbour_tables")[mode]
    checked = raised = 0
    for n, c, dist, row in comm_cases(mode):
        props = _props(n, mode, c, dist, row)
        want = got = None
        if LIVE:
            ref_props = ns.EnvironmentProperties(**_dump(props))
            random.seed(n * 1000 + c)
            try:
                d = Builder(ref_props.cluster_prop.agents_comm_prop, n).get_comm_link_list()
                want = [list(map(int, d[i])) for i in range(n)]
            except Exception as e:  # noqa: BLE001 -- the reference rejects (or trips over) the configuration
                want = type(e)
        else:
            want = tables[comm_key(n, c, dist, row)]
            want = Exception if want is None else want
        random.seed(n * 1000 + c)
        try:
            got = build_comm_table(props).tolist()
        except Exception as e:  # noqa: BLE001
            got = type(e)
        if isinstance(want, type):
            raised += 1
            # the reference fails: the drop-in must not silently produce a table either
            assert isinstance(got, type), (mode, n, c, dist, row, want, got)
        else:
            checked += 1
            assert got == want, (mode, n, c, dist, row)
    assert checked > 20


def test_random_sample_draw_matches_reference():
    from marl_demandresponse_b200.environment import random_sample_ids

    ns = refenv.load() if LIVE else None
    for n, c in SAMPLE_CASES:
        if LIVE:
            props = _props(n, "random_sample", c, 1, 5)
            ref_props = ns.EnvironmentProperties(**_dump(props))
            b = ns.comm_mod.AgentCommunicationBuilder(ref_props.cluster_prop.agents_comm_prop, n)
            random.seed(7)
            want = [list(map(int, b.get_random_sample(i))) for i in range(n)]
        else:
            want = stored("random_sample")[f"{n},{c}"]
        random.seed(7)
        got = [random_sample_ids(n, i, min(c, n - 1)) for i in range(n)]
        assert got == want


def test_default_property_tree_equals_reference_defaults():
    from marl_demandresponse_b200.properties import EnvironmentProperties

    ours = _dump(EnvironmentProperties())
    ref = _dump(refenv.load().EnvironmentProperties()) if LIVE else stored("default_properties")

    def walk(a, b, path):
        for k, v in b.items():
            assert k in a, f"missing default {path + k}"
            if isinstance(v, dict):
                walk(a[k], v, path + k + "/")
            elif isinstance(v, float):
                assert a[k] == pytest.approx(v, rel=0, abs=0), path + k
            else:
                assert str(a[k]) == str(v) or a[k] == v, (path + k, a[k], v)

    walk(ours, ref, "")


def test_perlin_wrapper_equals_reference_octave_sum():
    """``_Perlin`` (the drop-in's wrapper around the third-party generator) against the reference's
    ``Perlin.calculate_noise`` (perlin.py:41-56, last-octave weight quirk Q7) on the same generator --
    the deterministic stand-in both sides import, since ``perlin_noise`` is not a dependency of this project."""
    if LIVE:
        ns = refenv.load()
    else:
        refenv._install_stubs()
        want = stored("perlin")
    from marl_demandresponse_b200.environment import _Perlin

    for octaves, step, period, seed in PERLIN_CASES:
        ours = _Perlin(octaves, step, period, seed)
        assert ours.available
        if LIVE:
            ref = ns.perlin_mod.Perlin(1, octaves, step, period, seed)
            expect = [ref.calculate_noise(x) for x in PERLIN_X]
        else:
            expect = want[perlin_key(octaves, step, period, seed)]
        assert [ours.calculate_noise(x) for x in PERLIN_X] == expect


def test_interpolation_grids_equal_the_reference_files():
    """Key order and grids of the interpolation table: ``interp_dict_keys.csv:1`` /
    ``interp_parameters_dict.json:1`` against the generator's (``montecarlo.GRID``) and the oracle's."""
    import csv

    from marl_demandresponse_b200 import montecarlo
    from oracle.config import INTERP_GRIDS, INTERP_KEYS

    if LIVE:
        mc = os.path.join(refenv.REFERENCE_ROOT, "server/v0/monteCarlo")
        grids = json.load(open(os.path.join(mc, "interp_parameters_dict.json")))
        keys = [k.strip() for k in next(csv.reader(open(os.path.join(mc, "interp_dict_keys.csv")))) if k.strip()]
    else:
        keys, grids = stored("interp")["keys"], stored("interp")["grids"]
    assert keys == list(INTERP_KEYS) == list(montecarlo.KEYS)
    for k in keys:
        want = [float(v) for v in grids[k]]
        assert [float(v) for v in INTERP_GRIDS[k]] == want, k
        assert [float(v) for v in montecarlo.GRID[k]] == want, k


def greedy_cases(n):
    """Six seeded ``(t_air, target, cap, cop, lock, signal)`` observations of ``n`` houses."""
    rng = np.random.default_rng(n)
    for trial in range(6):
        target = 20.0 + np.abs(rng.normal(0, 1, n))
        t_air = target + rng.permutation(np.linspace(-3.0, 4.0, n))           # distinct differences
        cap = rng.choice([12500.0, 15000.0, 17500.0], n)
        cop = float(rng.choice([2.5, 2.3]))
        lock = rng.random(n) < 0.3
        signal = float(rng.uniform(0.0, 1.1) * (cap / cop).sum()) if trial else 0.0
        yield t_air, target, cap, cop, lock, signal


@pytest.mark.parametrize("n", GREEDY_N)
def test_greedy_myopic_restatement_equals_reference_controller(n):
    """``oracle.np_oracle.greedy_myopic`` (what ``k_greedy`` is compared with on the GPU) against the
    reference's ``GreedyMyopic.get_action`` (greedy_myopic_controller.py:67-104: pandas sort, first clause
    ignoring lock-out) on random observations with distinct temperatures (its sort is unstable on ties),
    over regulation signals from "nobody" to "everybody"."""
    from oracle.np_oracle import greedy_myopic

    if LIVE:
        gm = refenv.load_controller_module("greedy_myopic_controller")
    else:
        wants = stored("greedy_myopic")[str(n)]
    for trial, (t_air, target, cap, cop, lock, signal) in enumerate(greedy_cases(n)):
        if LIVE:
            obs = {i: {"indoor_temp": t_air[i], "target_temp": target[i], "cooling_capacity": cap[i], "cop": cop,
                       "lockout": bool(lock[i]), "reg_signal": signal} for i in range(n)}
            ctl = gm.GreedyMyopic({"id": 0}, None)
            ctl.get_action(obs)
            df = gm.GreedyMyopic.actions_df
            want = np.array([bool(df.loc[i]["HVAC_status"]) for i in range(n)])
        else:
            want = np.array(wants[trial], dtype=bool)
        got = np.asarray(greedy_myopic(t_air, target, cap, cop, lock, signal)).astype(bool)
        assert np.array_equal(got, want), (n, trial)


def bangbang_inputs():
    """``(t_air, target, deadband, on)`` of 400 seeded houses, the first 100 on the edges of the dead band."""
    rng = np.random.default_rng(3)
    n = 400
    target = 20.0 + np.abs(rng.normal(0, 1, n))
    db = rng.choice([0.0, 0.5, 1.0, 2.0], n)
    t_air = target + rng.uniform(-2, 2, n)
    t_air[:40] = target[:40] + db[:40] / 2        # on the upper edge
    t_air[40:80] = target[40:80] - db[40:80] / 2  # on the lower edge
    t_air[80:100] = target[80:100]                # exactly on target
    on = rng.random(n) < 0.5
    return t_air, target, db, on


def test_bangbang_rules_equal_reference_controllers():
    """``deadband_bangbang`` / ``bangbang`` of the oracle (the on-device policies are compared with them)
    against the reference's controller classes (bangbang_controllers.py:18-89), including the exact
    boundary values of the dead band."""
    import sys
    import types

    from oracle.np_oracle import bangbang, deadband_bangbang

    t_air, target, db, on = bangbang_inputs()
    n = len(t_air)
    ours = {"DeadbandBangBangController": deadband_bangbang(t_air, target, db, on),
            "BasicController": deadband_bangbang(t_air, target, db, on),
            "BangBangController": bangbang(t_air, target),
            "AlwaysOnController": np.ones(n, dtype=bool)}
    if LIVE:
        if "app.services.parser_service" not in sys.modules:   # only the type annotation MarlConfig is taken from it
            stub = types.ModuleType("app.services.parser_service")
            stub.MarlConfig = object
            sys.modules.setdefault("app.services", types.ModuleType("app.services"))
            sys.modules["app.services.parser_service"] = stub
        bb = refenv.load_controller_module("bangbang_controllers")
        obs = {i: {"indoor_temp": t_air[i], "target_temp": target[i], "deadband": db[i], "turned_on": bool(on[i])}
               for i in range(n)}
        wants = {name: [bool(getattr(bb, name)({"id": i}, None).act(obs)) for i in range(n)] for name in ours}
    else:
        wants = stored("bangbang")
    for name, got in ours.items():
        assert np.array_equal(np.asarray(got).astype(bool), np.array(wants[name], dtype=bool)), name


def _actor_probs(x, w):
    import torch

    h = torch.relu(x @ w[0][0].T + w[0][1])
    h = torch.relu(h @ w[1][0].T + w[1][1])
    return torch.softmax(h @ w[2][0].T + w[2][1], dim=1)


def test_actor_architecture_is_the_reference_actor():
    """The MA-PPO actor the tcgen05 kernel implements (Linear-ReLU-Linear-ReLU-Linear-softmax, probabilities
    over {off, on}; ``test_on_device_actor_matches_torch_fp32`` compares the kernel with exactly this
    computation) against the reference's ``Actor`` module (trainables/network.py:14-35) on its own weights."""
    import importlib.util
    import sys
    import types

    import torch

    if not LIVE:
        z = np.load(os.path.join(GOLDEN, "host_vs_reference", "actor.npz"))
        for j in range(len(ACTOR_CASES)):
            w = [(torch.from_numpy(z[f"w{j}_{i}"]), torch.from_numpy(z[f"b{j}_{i}"])) for i in range(3)]
            got = _actor_probs(torch.from_numpy(z[f"x{j}"]), w)
            assert got.shape == (37, 2) and torch.allclose(got, torch.from_numpy(z[f"p{j}"]), rtol=0, atol=1e-7)
        return
    if "app.utils.logger" not in sys.modules:   # pydantic BaseSettings moved: the logger module cannot load here
        stub = types.ModuleType("app.utils.logger")
        stub.logger = types.SimpleNamespace(info=lambda *a, **k: None, debug=lambda *a, **k: None)
        sys.modules["app.utils.logger"] = stub
    refenv.load()
    path = os.path.join(refenv.REFERENCE_ROOT, "server/app/core/agents/trainables/network.py")
    spec = importlib.util.spec_from_file_location("_ref_network", path)
    net = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(net)
    torch.manual_seed(0)
    for D, layers in ACTOR_CASES:
        actor = net.Actor(D, 2, layers)
        x = torch.randn(37, D)
        with torch.no_grad():
            want = actor(x)
            w = [(l.weight, l.bias) for l in actor.fc]
            assert len(w) == 3
            got = _actor_probs(x, w)
        assert got.shape == (37, 2) and torch.allclose(got, want, rtol=0, atol=1e-7)
