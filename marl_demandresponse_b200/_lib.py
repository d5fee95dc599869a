"""ctypes binding of ``libdrsim.so`` (the C ABI declared in ``include/drsim.h``).

There is no CPU fallback: importing this module loads the CUDA library or raises.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

ABI_VERSION = 4
MAX_SIGNAL_TERMS = 8
INTERP_SUBTABLES = 162
INTERP_SUBTABLE_LEN = 25920
N_METRICS = 6
N_ACC = 6
HALO_FIELDS = 8
SUMMARY_FIELDS = 8
REF_METRIC_FIELDS = 12

F32, F64 = 0, 1
PEN = {"individual_L2": 0, "common_L2": 1, "common_max_error": 2, "mixture": 3}
BASE = {"constant": 0, "interpolation": 1}
SIG = {"flat": 0, "sinusoidals": 1, "regular_steps": 2, "perlin": 3}
OBS = {"none": 0, "hand_engineered": 1, "tarmac": 2}
OBS_DTYPE = {"float32": 0, "bfloat16": 1}
COMM_RING, COMM_TABLE, COMM_SAMPLE = 0, 1, 2
MAX_SAMPLE_COMM = 32   # DRSIM_MAX_SAMPLE_COMM: nb_comm bound of the `random_sample` mode
NOISE = {"zero": 0, "philox": 1}
POLICY = {"external": 0, "deadband_bangbang": 1, "bangbang": 2, "always_on": 3, "greedy_myopic": 4}
PATH = {"auto": 0, "fused": 1, "split": 2}

_d, _i32, _i64, _u64 = C.c_double, C.c_int32, C.c_int64, C.c_uint64


class Config(C.Structure):
    """Mirror of ``drsim_config`` (field order and types must match include/drsim.h)."""

    _fields_ = [
        ("abi_version", _i32), ("n_rep", _i32), ("n_house", _i32), ("precision", _i32), ("dt", _i32), ("path", _i32),
        ("house_offset", _i64), ("n_house_global", _i64), ("rep_offset", _i64),
        ("deadband", _d), ("cop", _d), ("latent_cooling_fraction", _d),
        ("lockout_duration", _i32), ("solar_gain", _i32),
        ("window_area", _d), ("shading_coeff", _d), ("default_target_temp", _d),
        ("default_Ua", _d), ("default_Ca", _d), ("default_Cm", _d), ("default_Hm", _d),
        ("default_cooling_capacity", _d),
        ("day_temp", _d), ("night_temp", _d), ("temp_std", _d), ("phase", _d),
        ("alpha_temp", _d), ("alpha_sig", _d), ("norm_reg_sig", _d),
        ("penalty_mode", _i32), ("obs_dtype", _i32),
        ("alpha_ind_l2", _d), ("alpha_common_l2", _d), ("alpha_common_max", _d),
        ("base_power_mode", _i32), ("interp_update_period", _i32), ("interp_nb_agents", _i32), ("signal_mode", _i32),
        ("avg_power_per_hvac", _d),
        ("n_signal_terms", _i32), ("nb_octaves", _i32),
        ("amplitude_ratios", _d * MAX_SIGNAL_TERMS), ("periods", _d * MAX_SIGNAL_TERMS),
        ("amplitude_per_hvac", _d),
        ("octaves_step", _i32), ("period", _i32),
        ("obs_layout", _i32), ("nb_comm", _i32), ("comm_mode", _i32),
        ("state_solar_gain", _i32), ("state_thermal", _i32), ("state_hvac", _i32),
        ("message_thermal", _i32), ("message_hvac", _i32),
        ("noise_mode", _i32), ("policy", _i32),
        ("seed", _u64),
    ]


_pd, _pu8, _pi32, _pi64 = C.POINTER(_d), C.POINTER(C.c_uint8), C.POINTER(_i32), C.POINTER(_i64)


class HostState(C.Structure):
    _fields_ = [
        ("t_air", _pd), ("t_mass", _pd), ("target", _pd),
        ("Ua", _pd), ("Ca", _pd), ("Cm", _pd), ("Hm", _pd), ("cap", _pd),
        ("on", _pu8), ("lockout", _pu8), ("sso", _pi32), ("epoch", _pi64),
        ("od_temp", _pd), ("signal", _pd), ("base_power", _pd), ("power", _pd), ("solar", _pd),
        ("artificial_ratio", _pd), ("max_power", _pd), ("t_since_interp", _pi32),
        ("thermal_coefs", _pd), ("lockout_duration", _pi32),
    ]


class RolloutSlot(C.Structure):
    """Mirror of ``drsim_rollout_slot``."""
    _fields_ = [("obs", C.c_void_p), ("actions", C.c_void_p), ("prob", C.c_void_p), ("reward", C.c_void_p),
                ("next_obs", C.c_void_p)]


class SnapshotView(C.Structure):
    """Mirror of ``drsim_snapshot_view``."""
    _fields_ = [("n_rep", _i32), ("n_house", _i32), ("obs_dim", _i32), ("real_bytes", _i32),
                ("t_air", _pd), ("t_mass", _pd), ("reward", _pd), ("sso", _pi32), ("on", _pu8), ("lockout", _pu8),
                ("env", _pd), ("obs", C.c_void_p)]


class ActorNet(C.Structure):
    """Mirror of ``drsim_actor_net``."""

    _fields_ = [("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w3", C.c_void_p), ("b3", C.c_void_p), ("h1", C.c_int32), ("h2", C.c_int32),
                ("precision", C.c_int32), ("pad_", C.c_int32)]


class Ptrs(C.Structure):
    _fields_ = [
        ("n_rep", _i32), ("n_house", _i32), ("house_stride", _i32), ("obs_dim", _i32), ("real_bytes", _i32),
        ("nb_comm", _i32), ("temp_is_deviation", _i32), ("obs_bytes", _i32),
        ("t_air", C.c_void_p), ("t_mass", C.c_void_p), ("sso", C.c_void_p), ("flags", C.c_void_p),
        ("target", C.c_void_p), ("cap", C.c_void_p), ("reward", C.c_void_p), ("obs", C.c_void_p),
        ("actions", C.c_void_p), ("epoch", C.c_void_p),
        ("od_temp", C.c_void_p), ("signal", C.c_void_p), ("base_power", C.c_void_p), ("power", C.c_void_p),
        ("solar", C.c_void_p), ("pen_sum", C.c_void_p), ("pen_max", C.c_void_p),
        ("comm_table", C.c_void_p), ("metrics", C.c_void_p), ("acc", C.c_void_p), ("rew_sig", C.c_void_p),
        ("halo_out", C.c_void_p),
    ]


class StepArgs(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("od_noise", C.c_void_p), ("perlin", C.c_void_p), ("interp_ids", C.c_void_p)]


class ResetArgs(C.Structure):
    _fields_ = [("seed", _u64), ("mode", _i32), ("randomize_date", _i32), ("start_epoch", _i64),
                ("init_air_temp", _d), ("init_mass_temp", _d), ("std_target_temp", _d),
                ("factor_low", _d), ("factor_high", _d), ("quirk_ua", _i32), ("n_caps", _i32), ("caps", _d * 8)]


class DrsimError(RuntimeError):
    pass


_lib = None


def lib():
    """Load (building first if the in-tree library is missing or stale) and bind the C ABI."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path) or (_build.stale() and os.environ.get("DRSIM_NO_REBUILD") != "1"):
        try:
            _build.build()
        except Exception as e:  # noqa: BLE001
            if not os.path.exists(path):
                raise DrsimError(f"libdrsim.so is not built and cannot be built here ({e}); "
                                 "the CUDA extension is mandatory -- there is no CPU fallback") from e
    L = C.CDLL(path)
    hp = C.c_void_p
    sig = {
        "drsim_create": (C.c_int, [C.POINTER(Config), C.c_int, C.POINTER(hp)]),
        "drsim_destroy": (C.c_int, [hp]),
        "drsim_clone": (C.c_int, [hp, C.POINTER(hp)]),
        "drsim_buffers": (C.c_int, [hp, C.POINTER(Ptrs)]),
        "drsim_set_state": (C.c_int, [hp, C.POINTER(HostState), C.c_void_p]),
        "drsim_get_state": (C.c_int, [hp, C.POINTER(HostState), C.c_void_p]),
        "drsim_reset": (C.c_int, [hp, C.POINTER(ResetArgs), C.c_void_p]),
        "drsim_set_comm_table": (C.c_int, [hp, C.c_void_p, C.c_int, C.c_void_p]),
        "drsim_set_interp_table": (C.c_int, [hp, C.c_void_p, C.c_void_p]),
        "drsim_comm_sample": (C.c_int, [hp, _i64, C.c_void_p, C.c_void_p]),
        "drsim_step_count": (C.c_int64, [hp]),
        "drsim_step": (C.c_int, [hp, C.POINTER(StepArgs), C.c_void_p]),
        "drsim_run": (C.c_int, [hp, C.POINTER(StepArgs), C.c_int, C.c_size_t, C.c_void_p]),
        "drsim_run_tape": (C.c_int, [hp, C.POINTER(StepArgs), C.c_int, C.c_size_t, C.c_int, C.c_void_p]),
        "drsim_refresh": (C.c_int, [hp, C.POINTER(StepArgs), C.c_int, C.c_void_p]),
        "drsim_step_begin": (C.c_int, [hp, C.POINTER(StepArgs), C.c_void_p]),
        "drsim_step_finish": (C.c_int, [hp, C.POINTER(StepArgs), C.c_void_p, C.c_int, C.c_void_p]),
        "drsim_step_sharded": (C.c_int, [hp, C.POINTER(StepArgs), C.c_void_p]),
        "drsim_step_finish_gathered": (C.c_int, [hp, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
        "drsim_ipc_export": (C.c_int, [hp, C.c_void_p]),
        "drsim_ipc_attach": (C.c_int, [hp, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
        "drsim_peer_status": (C.c_int, [hp, C.c_void_p]),
        "drsim_peer_attach_local": (C.c_int, [C.POINTER(hp), C.c_int, C.c_void_p]),
        "drsim_step_host": (C.c_int, [hp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
        "drsim_step_host_full": (C.c_int, [hp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
        "drsim_snapshot": (C.c_int, [hp, C.POINTER(SnapshotView), C.c_void_p]),
        "drsim_step_host_snapshot": (C.c_int, [hp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SnapshotView),
                                               C.c_void_p]),
        "drsim_policy_step": (C.c_int, [hp, C.POINTER(ActorNet), _u64, C.c_void_p, C.c_void_p, C.c_void_p]),
        "drsim_rollout_transition": (C.c_int, [hp, C.POINTER(ActorNet), _u64, C.POINTER(RolloutSlot), C.c_void_p]),
        "drsim_launch_count": (C.c_int64, [hp]),
        "drsim_fused_info": (C.c_int, [hp, C.POINTER(_i32 * 6)]),
        "drsim_step_route": (C.c_int, [hp]),
        "drsim_cluster_summary": (C.c_int, [hp, C.c_void_p, C.c_void_p]),
        "drsim_metrics_update": (C.c_int, [hp, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
        "drsim_host_solar_gain": (C.c_double, [_i64, _d, _d]),
        "drsim_host_od_temp": (C.c_double, [_i64, _d, _d, _d, _d]),
        "drsim_host_civil": (None, [_i64, C.POINTER(_i32 * 7)]),
        "drsim_host_thermal_coefs": (None, [_d, _d, _d, _d, _i32, C.POINTER(_d * 12)]),
        "drsim_host_philox": (None, [_u64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32 * 4)]),
        "drsim_host_comm_sample": (None, [_u64, _i64, _i64, _i64, _i64, C.c_int, C.c_void_p]),
        "drsim_last_error": (C.c_char_p, []),
        "drsim_abi_version": (C.c_int, []),
        "drsim_sizeof": (C.c_int, [C.c_int]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.drsim_abi_version() != ABI_VERSION:
        raise DrsimError("libdrsim.so ABI version mismatch")
    for which, st in enumerate((Config, HostState, Ptrs, StepArgs, ResetArgs)):
        if L.drsim_sizeof(which) != C.sizeof(st):
            raise DrsimError(f"struct layout mismatch for {st.__name__}: C {L.drsim_sizeof(which)} vs ctypes {C.sizeof(st)}")
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "drsim_create", "drsim_destroy", "drsim_clone", "drsim_buffers", "drsim_set_state", "drsim_get_state", "drsim_reset",
    "drsim_set_comm_table", "drsim_set_interp_table", "drsim_step", "drsim_run", "drsim_run_tape", "drsim_refresh", "drsim_step_begin",
    "drsim_step_finish", "drsim_step_sharded", "drsim_step_finish_gathered", "drsim_step_host", "drsim_step_host_full", "drsim_snapshot", "drsim_step_host_snapshot",
    "drsim_ipc_export", "drsim_ipc_attach", "drsim_peer_status", "drsim_peer_attach_local", "drsim_policy_step", "drsim_rollout_transition", "drsim_launch_count", "drsim_fused_info", "drsim_step_route", "drsim_cluster_summary", "drsim_metrics_update", "drsim_host_solar_gain", "drsim_host_od_temp",
    "drsim_host_civil", "drsim_host_thermal_coefs", "drsim_host_philox", "drsim_last_error", "drsim_abi_version",
    "drsim_sizeof", "drsim_comm_sample", "drsim_step_count", "drsim_host_comm_sample",
]


def check(rc: int) -> None:
    if rc != 0:
        raise DrsimError(f"libdrsim error {rc}: {lib().drsim_last_error().decode()}")
