"""CPU-side checks of the C ABI: the library loads, exports every declared symbol, struct
layouts agree, and the __host__ __device__ env-level code matches the oracle."""
import ctypes as C
import datetime as dt
import os
import re

import numpy as np
import pytest

from marl_demandresponse_b200 import _lib
from oracle import np_oracle, philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    header = open(os.path.join(ROOT, "include", "drsim.h")).read()
    declared = set(re.findall(r"\b(drsim_[a-z_0-9]+)\s*\(", header))
    declared -= {"drsim_t"}
    assert declared, "no prototypes parsed"
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/drsim.h but not exported"
    assert set(_lib.EXPORTED_SYMBOLS) == declared


def test_struct_layouts_match():
    L = _lib.lib()
    for which, st in enumerate((_lib.Config, _lib.HostState, _lib.Ptrs, _lib.StepArgs, _lib.ResetArgs)):
        assert L.drsim_sizeof(which) == C.sizeof(st)


def test_create_fails_loudly_without_gpu_or_on_bad_config():
    import torch

    L = _lib.lib()
    cfg = _lib.Config()
    h = C.c_void_p()
    rc = L.drsim_create(C.byref(cfg), 0, C.byref(h))  # abi_version = 0
    assert rc == -1 and b"abi_version" in L.drsim_last_error()
    if not torch.cuda.is_available():
        from marl_demandresponse_b200 import flatten_config

        cfg = flatten_config(None, 1)
        rc = L.drsim_create(C.byref(cfg), 0, C.byref(h))
        assert rc != 0 and not h.value, "must not fall back to a CPU path"


def test_house_sharded_greedy_myopic_is_refused():
    """Greedy-myopic sorts the whole cluster against the cluster's signal: a handle holding part of the houses refuses
    it before it looks for a device (each shard would fill the whole signal on its own)."""
    from marl_demandresponse_b200 import flatten_config

    L = _lib.lib()
    h = C.c_void_p()
    p = {"cluster_prop": {"nb_agents": 64}}
    cfg = flatten_config(p, 2, "f32", "tarmac", policy="greedy_myopic", path="split", house_offset=32, n_house_local=32)
    assert cfg.policy == _lib.POLICY["greedy_myopic"]
    rc = L.drsim_create(C.byref(cfg), 0, C.byref(h))
    msg = L.drsim_last_error().decode()
    assert rc == -1 and not h.value and "house-sharded cluster: the greedy scan sorts the whole cluster" in msg, (rc, msg)


def _epochs():
    rng = np.random.default_rng(3)
    base = np_oracle.to_epoch(dt.datetime(2019, 1, 1))
    e = list(base + rng.integers(0, 8 * 366 * 86400, 400))
    for s in ("2024-02-29T07:29:59", "2024-02-29T07:30:00", "2021-06-15T17:30:00", "2021-06-15T17:31:00",
              "2023-12-31T23:59:59", "2024-01-01T00:00:00", "2000-02-29T12:00:00", "2100-03-01T00:00:00",
              "1970-01-01T00:00:00"):
        e.append(np_oracle.to_epoch(dt.datetime.fromisoformat(s)))
    return [int(x) for x in e]


def test_civil_solar_odtemp_match_oracle():
    L = _lib.lib()
    out = (C.c_int32 * 7)()
    tp = {"day_temp": 31.0, "night_temp": 19.5, "phase": 1.5}
    for e in _epochs():
        d = np_oracle.from_epoch(e)
        L.drsim_host_civil(e, C.byref(out))
        assert list(out) == [d.year, d.month, d.day, d.hour, d.minute, d.second, d.timetuple().tm_yday]
        want = np_oracle.solar_gain_scalar(d, 7.175, 0.67)
        got = L.drsim_host_solar_gain(e, 7.175, 0.67)
        assert abs(got - want) <= 1e-12 * max(1.0, abs(want))
        want = np_oracle.od_temp_scalar(d, tp, 0.37)
        got = L.drsim_host_od_temp(e, tp["day_temp"], tp["night_temp"], tp["phase"], 0.37)
        assert abs(got - want) <= 1e-13 * 30


def test_thermal_coefficients_reproduce_the_literal_update():
    """fp32-path difference form == building.py:141-222 literal update (evaluated in fp64)."""
    L = _lib.lib()
    rng = np.random.default_rng(5)
    out = (C.c_double * 12)()
    for _ in range(200):
        Ua = rng.choice([218.0 * rng.uniform(0.9, 1.1), rng.uniform(0.9, 1.1)])  # with / without quirk Q1
        Ca, Cm, Hm = 9.08e5 * rng.uniform(0.9, 1.1), 3.45e6 * rng.uniform(0.9, 1.1), 2.84e3 * rng.uniform(0.9, 1.1)
        dt_s = int(rng.choice([1, 4, 7, 60]))
        L.drsim_host_thermal_coefs(Ua, Ca, Cm, Hm, dt_s, C.byref(out))
        c = np.array(out[:6])
        ta, tm, od = rng.uniform(15, 30), rng.uniform(15, 30), rng.uniform(10, 40)
        Qa = rng.choice([0.0, -15000 / 1.35]) + rng.uniform(0, 800)
        na, nm = np_oracle.thermal_update(ta, tm, Ua, Ca, Cm, Hm, od, Qa, dt_s)
        ga = ta + c[0] * (tm - ta) + c[1] * (od - ta) + c[2] * Qa
        gm = tm + c[3] * (ta - tm) + c[4] * (od - tm) + c[5] * Qa
        assert abs(ga - na) < 2e-10 and abs(gm - nm) < 2e-10, (ga - na, gm - nm)


def test_philox_matches_numpy_restatement():
    L = _lib.lib()
    out = (C.c_uint32 * 4)()
    rng = np.random.default_rng(7)
    # known-answer vectors of Random123 (philox4x32-10, kat_vectors): counter, key -> output
    L.drsim_host_philox(0, 0, 0, 0, 0, C.byref(out))
    assert [hex(v) for v in out] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    L.drsim_host_philox(0xFFFFFFFFFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, C.byref(out))
    assert [hex(v) for v in out] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    L.drsim_host_philox((0x299F31D0 << 32) | 0xA4093822, 0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, C.byref(out))
    assert [hex(v) for v in out] == ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]
    for _ in range(50):
        key = int(rng.integers(0, 2**63))
        c = [int(x) for x in rng.integers(0, 2**32, 4)]
        L.drsim_host_philox(key, *c, C.byref(out))
        want = philox.philox4x32_10(key, *c)
        assert [int(v) for v in out] == [int(w) for w in want]


def test_v0_config_translation_and_norm_vector():
    """Legacy config_dict -> app-style property tree (no GPU needed), and the legacy normStateDict
    restatement on a hand-made observation dict (v0/utils.py:541-657: float lock-out ratio, power over
    norm_reg_sig * nb_agents)."""
    import datetime as dt
    import json
    import os

    import numpy as np

    from marl_demandresponse_b200.v0 import norm_state_dict_v0, props_from_v0

    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "v0_n20_sinus_mixture_flags.npz"))
    cfg = json.loads(str(z["config_json"]))
    p = props_from_v0(cfg)
    assert p.cluster_prop.nb_agents == 20 and p.cluster_prop.agents_comm_prop.mode == "closed_groups"
    assert p.cluster_prop.agents_comm_prop.max_nb_agents_communication == 4
    assert p.power_grid_prop.signal_properties.mode == "sinusoidals" and p.reward_prop.penalty_props.mode == "mixture"
    assert p.cluster_prop.house_prop.hvac_prop.noise_prop.cooling_capacity_list == [12500, 15000, 17500]
    assert p.time_step == dt.timedelta(seconds=4) and p.start_datetime_mode == "random"
    obs = {"house_temp": 22.0, "house_mass_temp": 21.0, "house_target_temp": 20.0, "house_deadband": 0.0, "OD_temp": 30.0,
           "house_solar_gain": 500.0, "hvac_cooling_capacity": 15000, "house_Ua": 218.0, "house_Cm": 3.45e6, "house_Ca": 9.08e5,
           "house_Hm": 2840.0, "hvac_COP": 2.5, "hvac_latent_cooling_fraction": 0.35, "hvac_turned_on": True, "hvac_lockout": False,
           "hvac_seconds_since_off": 12, "hvac_lockout_duration": 40, "reg_signal": 75000.0, "cluster_hvac_power": 30000.0,
           "datetime": dt.datetime(2021, 1, 1), "message": []}
    d = norm_state_dict_v0(obs, cfg, return_dict=True)
    assert d["hvac_seconds_since_off"] == 0.3 and d["house_temp"] == 0.4 and d["OD_temp"] == 2.0
    assert d["cluster_hvac_power"] == 30000.0 / (7500 * 20) and d["reg_signal"] == 0.5 and d["house_solar_gain"] == 0.5
    assert norm_state_dict_v0(obs, cfg).shape == (len(d) - 1,)
