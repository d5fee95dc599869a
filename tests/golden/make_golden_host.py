"""Generate ``tests/golden/host_vs_reference/`` (``values.json``, ``actor.npz``): the values the host-side
reference comparisons (``tests/test_host_vs_reference.py``, ``tests/test_montecarlo_vs_reference.py``) check
against, so that they also run where the reference checkout is absent.

    python tests/golden/make_golden_host.py

The values are those of this project's implementation on exactly the inputs on which the live comparisons with
the running reference assert equality (neighbour tables, sample ids, defaults, Perlin sums, grids and controller
decisions bit for bit; the Monte-Carlo entries to 1e-9) and passed (DESIGN.md section 2), so they stand for the
reference's values there.  The actor file holds fixed weights, inputs and the probabilities of the
Linear-ReLU-Linear-ReLU-Linear-softmax forward on them.  ``source`` in the JSON file records where they came from.
"""
from __future__ import annotations

import json
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import test_host_vs_reference as T  # noqa: E402  (the case lists of the tests themselves)
import test_montecarlo_vs_reference as M  # noqa: E402


def neighbour_tables() -> dict:
    from marl_demandresponse_b200.environment import build_comm_table

    out = {}
    for mode in T.COMM_MODES:
        tables = {}
        for n, c, dist, row in T.comm_cases(mode):
            random.seed(n * 1000 + c)
            try:
                tables[T.comm_key(n, c, dist, row)] = build_comm_table(T._props(n, mode, c, dist, row)).tolist()
            except Exception:  # noqa: BLE001 -- the reference raises on these configurations
                tables[T.comm_key(n, c, dist, row)] = None
        out[mode] = tables
    return out


def random_samples() -> dict:
    from marl_demandresponse_b200.environment import random_sample_ids

    out = {}
    for n, c in T.SAMPLE_CASES:
        random.seed(7)
        out[f"{n},{c}"] = [list(map(int, random_sample_ids(n, i, min(c, n - 1)))) for i in range(n)]
    return out


def default_properties() -> dict:
    from marl_demandresponse_b200.properties import EnvironmentProperties

    return json.loads(json.dumps(T._dump(EnvironmentProperties()), default=str))


def perlin() -> dict:
    from marl_demandresponse_b200.environment import _Perlin
    from oracle import refenv

    refenv._install_stubs()   # the deterministic stand-in for perlin_noise both sides use
    return {T.perlin_key(*p): [_Perlin(*p).calculate_noise(x) for x in T.PERLIN_X] for p in T.PERLIN_CASES}


def interp_grids() -> dict:
    from oracle.config import INTERP_GRIDS, INTERP_KEYS

    return {"keys": list(INTERP_KEYS), "grids": {k: [float(v) for v in INTERP_GRIDS[k]] for k in INTERP_KEYS}}


def greedy() -> dict:
    from oracle.np_oracle import greedy_myopic

    return {str(n): [np.asarray(greedy_myopic(*case)).astype(bool).tolist() for case in T.greedy_cases(n)]
            for n in T.GREEDY_N}


def bangbang() -> dict:
    from oracle.np_oracle import bangbang as bb, deadband_bangbang

    t_air, target, db, on = T.bangbang_inputs()
    n = len(t_air)
    dbb = np.asarray(deadband_bangbang(t_air, target, db, on)).astype(bool).tolist()
    return {"DeadbandBangBangController": dbb, "BasicController": dbb,
            "BangBangController": np.asarray(bb(t_air, target)).astype(bool).tolist(),
            "AlwaysOnController": [True] * n}


def montecarlo() -> dict:
    from marl_demandresponse_b200 import montecarlo as mc
    from oracle.montecarlo import table_entries

    idx = M.grid_indices()
    prop = mc.env_prop_for_table()
    house = {k: v for k, v in prop["cluster_prop"]["house_prop"].items() if k != "hvac_prop"}
    pts = mc.grid_points(idx)
    return {"indices": idx.tolist(), "house": house,
            "values": table_entries(prop, mc.initial_state(pts, prop), pts["OD_temp"]).tolist()}


def actor() -> dict:
    import torch

    torch.manual_seed(0)
    out = {}
    for j, (D, layers) in enumerate(T.ACTOR_CASES):
        widths = [D] + (json.loads(layers) if isinstance(layers, str) else list(layers)) + [2]
        fc = [torch.nn.Linear(a, b) for a, b in zip(widths[:-1], widths[1:])]
        x = torch.randn(37, D)
        with torch.no_grad():
            h = x
            for i, lin in enumerate(fc):
                h = lin(h)
                h = torch.relu(h) if i < len(fc) - 1 else torch.softmax(h, dim=1)
        out[f"x{j}"] = x.numpy()
        out[f"p{j}"] = h.numpy()
        for i, lin in enumerate(fc):
            out[f"w{j}_{i}"] = lin.weight.detach().numpy()
            out[f"b{j}_{i}"] = lin.bias.detach().numpy()
    return out


def main():
    data = {
        "source": "this project's implementation, on inputs where the live comparisons assert it equals the reference",
        "neighbour_tables": neighbour_tables(), "random_sample": random_samples(),
        "default_properties": default_properties(), "perlin": perlin(), "interp": interp_grids(),
        "greedy_myopic": greedy(), "bangbang": bangbang(), "montecarlo": montecarlo(),
    }
    with open(os.path.join(HERE, "host_vs_reference", "values.json"), "w") as f:
        json.dump(data, f, separators=(",", ":"))
    np.savez_compressed(os.path.join(HERE, "host_vs_reference", "actor.npz"), **actor())


if __name__ == "__main__":
    main()
