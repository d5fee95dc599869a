"""The Monte-Carlo table restatement (``oracle/montecarlo.py``, and the host-side state builder of the
GPU generator, ``marl_demandresponse_b200/montecarlo.py``) against the reference's own point evaluator.

``server/v0/monteCarlo/monteCarlo.py`` runs its whole 4.2 M-point sweep at import time, so only its
``eval_parameters_bangbang_average_consumption`` (:152-230) is taken -- parsed out of the file and executed
with the real legacy env, controller and config as its globals -- and evaluated on a handful of random
grid points.  Authoring container only (needs ``/root/reference``); the GPU generator is compared with the
same restatement in ``test_monte_carlo_table_generator_matches_oracle``.  Without the reference checkout the
restatement is compared with the evaluator's values on the same points, stored in
``tests/golden/host_vs_reference/values.json`` (``tests/golden/make_golden_host.py``).
"""
import ast
import copy
import datetime
import json
import os
import random
import sys
import types

import numpy as np
import pytest

from oracle import refenv

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)


def grid_indices():
    """24 seeded grid points plus the corners: first / last entry, a midnight and an end-of-year point."""
    rng = np.random.default_rng(5)
    idx = np.sort(rng.choice(4_199_040, size=24, replace=False))
    return np.unique(np.concatenate([idx, [0, 4_199_039, 5, 71]]))


def reference_point_evaluator():
    import make_golden_v0 as g

    saved = {k: sys.modules.get(k) for k in ("matplotlib", "matplotlib.pyplot", "perlin_noise")}
    try:
        config_dict, Env, _ = g.load_v0()
        v0_dir = os.path.join(refenv.REFERENCE_ROOT, "server", "v0")
        if "v0.agents" not in sys.modules:   # the package __init__ pulls in every trainer (torch, cvxpy, ...)
            pkg = types.ModuleType("v0.agents")
            pkg.__path__ = [os.path.join(v0_dir, "agents")]
            sys.modules["v0.agents"] = pkg
        from v0.agents.bangbang_controllers import BangBangController
        from v0.utils import get_actions
    finally:
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
            else:
                sys.modules.pop(k, None)
    path = os.path.join(v0_dir, "monteCarlo", "monteCarlo.py")
    tree = ast.parse(open(path).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "eval_parameters_bangbang_average_consumption")
    def get_actions_legacy_keys(actors, obs_dict):
        # As shipped, the legacy controller reads the app's key names (bangbang_controllers.py:50-51:
        # "indoor_temp", "target_temp") while the legacy env emits "house_temp" / "house_target_temp"
        # (MA_DemandResponse.py:888-917) -- the script raises KeyError unmodified.  The two keys are aliased
        # here; the controller, the env and the averaging loop are the reference's own.
        view = {i: dict(o, indoor_temp=o["house_temp"], target_temp=o["house_target_temp"]) for i, o in obs_dict.items()}
        return get_actions(actors, view)

    scope = dict(copy=copy, datetime=datetime, timedelta=datetime.timedelta, config_dict=config_dict, MADemandResponseEnv=Env,
                 BangBangController=BangBangController, get_actions=get_actions_legacy_keys, d0=datetime.date(2021, 1, 1),
                 NB_TIME_STEPS_BY_SIM=75, NB_TIME_STEPS_AVG=10)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), scope)
    return scope[fn.name], config_dict


def test_table_restatement_matches_reference_point_evaluator():
    from marl_demandresponse_b200 import montecarlo as mc
    from oracle.montecarlo import table_entries

    idx = grid_indices()
    pts = mc.grid_points(idx)
    if not refenv.available():
        with open(os.path.join(GOLDEN, "host_vs_reference", "values.json")) as f:
            g = json.load(f)["montecarlo"]
        assert g["indices"] == idx.tolist()
        prop = mc.env_prop_for_table(g["house"])
        got = table_entries(prop, mc.initial_state(pts, prop), pts["OD_temp"])
        np.testing.assert_allclose(got, np.asarray(g["values"], dtype=np.float64), rtol=1e-9, atol=1e-6)
        assert np.ptp(got) > 100.0
        return
    evaluate, config_dict = reference_point_evaluator()
    house = {k: config_dict["default_house_prop"][k] for k in ("Ua", "Ca", "Cm", "Hm", "target_temp", "deadband", "window_area",
                                                               "shading_coeff", "solar_gain_bool") if k in config_dict["default_house_prop"]}
    if "solar_gain_bool" in house:
        house["solar_gain"] = house.pop("solar_gain_bool")
    prop = mc.env_prop_for_table(house)
    hv, dflt = prop["cluster_prop"]["house_prop"]["hvac_prop"], config_dict["default_hvac_prop"]
    assert hv["cop"] == dflt["COP"] and hv["latent_cooling_fraction"] == dflt["latent_cooling_fraction"]
    want = []
    state = random.getstate()
    try:
        for j in range(len(idx)):
            want.append(evaluate(**{k: (float(pts[k][j]) if k not in ("date",) else int(pts[k][j])) for k in mc.KEYS}))
    finally:
        random.setstate(state)
    got = table_entries(prop, mc.initial_state(pts, prop), pts["OD_temp"])
    np.testing.assert_allclose(got, np.asarray(want, dtype=np.float64), rtol=1e-9, atol=1e-6)
    assert np.ptp(got) > 100.0   # the sample is not degenerate (different duty cycles)
