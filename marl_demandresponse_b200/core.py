"""Thin Python owner of a ``drsim_t`` handle: config flattening, state I/O, zero-copy views.

PyTorch is used only as plumbing (device tensors aliasing the library's buffers, the current
CUDA stream); all arithmetic of the step happens in ``libdrsim.so``.
"""
from __future__ import annotations

import ctypes as C
import datetime as _dt
from typing import Any, Dict, Optional

import numpy as np

from . import _lib
from .properties import EnvironmentProperties, as_props

EPOCH0 = _dt.datetime(1970, 1, 1)


def to_epoch(dt: _dt.datetime) -> int:
    d = dt - EPOCH0
    return d.days * 86400 + d.seconds


def from_epoch(sec: int) -> _dt.datetime:
    return EPOCH0 + _dt.timedelta(seconds=int(sec))


def nb_comm_of(props: EnvironmentProperties) -> int:
    """agent_communication_builder.py:49-52."""
    cp = props.cluster_prop
    return int(min(cp.agents_comm_prop.max_nb_agents_communication, cp.nb_agents - 1))


def comm_width(props: EnvironmentProperties) -> int:
    """Number of neighbour messages per agent = width of the table the reference builds:
    ``neighbours`` / ``random_*``: nb_comm; ``closed_groups``: the un-clamped
    ``max_nb_agents_communication`` when the first group is complete
    (agent_communication_builder.py:94-101); ``neighbours_2D``: 2 d (d + 1) cells of the
    Manhattan ball (:152-166), independent of nb_comm."""
    cp = props.cluster_prop.agents_comm_prop
    c = nb_comm_of(props)
    if cp.mode == "neighbours_2D":
        d = cp.max_communication_distance
        return 2 * d * (d + 1)
    if cp.mode == "closed_groups" and c <= props.cluster_prop.nb_agents:
        return cp.max_nb_agents_communication if c == cp.max_nb_agents_communication else c
    return c


def flatten_config(props: Any, n_rep: int = 1, precision: str = "f32", obs_layout: str = "hand_engineered",
                   policy: str = "external", noise: str = "zero", seed: int = 0, path: str = "auto",
                   comm_table: bool | None = None, house_offset: int = 0, n_house_local: int | None = None,
                   rep_offset: int = 0, obs_dtype: str = "float32") -> _lib.Config:
    """``EnvironmentProperties`` -> ``drsim_config`` (include/drsim.h).  ``obs_dtype``: element type of the
    observation rows, "float32" (the build's precision) or "bfloat16" (fp32 build only: every row element is the
    fp32 value rounded to nearest-even)."""
    if obs_dtype not in _lib.OBS_DTYPE:
        raise ValueError(f"obs_dtype must be one of {sorted(_lib.OBS_DTYPE)}, got {obs_dtype!r}")
    p = as_props(props)
    hp, hv = p.cluster_prop.house_prop, p.cluster_prop.house_prop.hvac_prop
    gp, rp = p.power_grid_prop, p.reward_prop
    sp, bp = gp.signal_properties, gp.base_power_props
    c = _lib.Config()
    c.abi_version = _lib.ABI_VERSION
    c.n_rep = int(n_rep)
    n_glob = int(p.cluster_prop.nb_agents)
    c.n_house = int(n_house_local) if n_house_local is not None else n_glob
    c.house_offset = int(house_offset)
    c.n_house_global = n_glob
    c.rep_offset = int(rep_offset)
    c.precision = {"f32": _lib.F32, "f64": _lib.F64}[precision]
    c.dt = int(p.time_step.seconds)  # hvac.py:46 reads time_step.seconds
    c.path = _lib.PATH[path]
    c.deadband = hp.deadband
    c.cop = hv.cop
    c.latent_cooling_fraction = hv.latent_cooling_fraction
    c.lockout_duration = hv.lockout_duration
    c.solar_gain = int(hp.solar_gain)
    c.window_area = hp.window_area
    c.shading_coeff = hp.shading_coeff
    c.default_target_temp = hp.target_temp
    c.default_Ua, c.default_Ca, c.default_Cm, c.default_Hm = hp.Ua, hp.Ca, hp.Cm, hp.Hm
    c.default_cooling_capacity = hv.cooling_capacity
    tp = p.temp_prop
    c.day_temp, c.night_temp, c.temp_std, c.phase = tp.day_temp, tp.night_temp, tp.temp_std, tp.phase
    c.alpha_temp, c.alpha_sig, c.norm_reg_sig = rp.alpha_temp, rp.alpha_sig, float(rp.norm_reg_sig)
    c.penalty_mode = _lib.PEN[rp.penalty_props.mode]
    c.alpha_ind_l2 = rp.penalty_props.alpha_ind_l2
    c.alpha_common_l2 = rp.penalty_props.alpha_common_l2
    c.alpha_common_max = rp.penalty_props.alpha_common_max
    if rp.sig_penalty_mode != "common_L2":  # rewards_calculator.py:197-201
        raise ValueError(f"Unknown signal penalty mode: {rp.sig_penalty_mode}")
    c.base_power_mode = _lib.BASE[bp.mode]
    c.interp_update_period = bp.interp_update_period
    c.interp_nb_agents = bp.interp_nb_agents
    c.avg_power_per_hvac = float(bp.avg_power_per_hvac)
    c.signal_mode = _lib.SIG[sp.mode]
    if sp.mode == "sinusoidals" and len(sp.periods) != len(sp.amplitude_ratios):
        raise ValueError(  # signal_calculator.py:61-66
            "Power grid signal parameters: periods and amplitude_ratios lists should have the same length.")
    n_terms = min(len(sp.amplitude_ratios), _lib.MAX_SIGNAL_TERMS)
    c.n_signal_terms = n_terms
    for k in range(n_terms):
        c.amplitude_ratios[k] = sp.amplitude_ratios[k]
        if k < len(sp.periods):
            c.periods[k] = float(sp.periods[k])
    c.amplitude_per_hvac = float(sp.amplitude_per_hvac)
    c.nb_octaves, c.octaves_step, c.period = sp.nb_octaves, sp.octaves_step, sp.period
    c.obs_layout = _lib.OBS[obs_layout]
    c.obs_dtype = _lib.OBS_DTYPE[obs_dtype]
    c.nb_comm = comm_width(p)
    mode = p.cluster_prop.agents_comm_prop.mode
    if comm_table is None and mode == "random_sample":
        c.comm_mode = _lib.COMM_SAMPLE     # drawn on the device every step (drsim_comm_sample)
    else:
        if comm_table is None:
            comm_table = mode != "neighbours"
        c.comm_mode = _lib.COMM_TABLE if comm_table else _lib.COMM_RING
    st, mp = p.state_prop, p.cluster_prop.message_prop
    c.state_solar_gain, c.state_thermal, c.state_hvac = int(st.solar_gain), int(st.thermal), int(st.hvac)
    c.message_thermal, c.message_hvac = int(mp.thermal), int(mp.hvac)
    c.noise_mode = _lib.NOISE[noise]
    c.policy = _lib.POLICY[policy]
    c.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return c


def thermal_coefs(Ua, Ca, Cm, Hm, dt: int) -> np.ndarray:
    """Vectorised fp64 derivation of the per-house update constants (building.py:186-206), laid
    out as ``drsim_host_thermal_coefs`` does: [..., 0:6] difference-form coefficients of the fp32
    path, [..., 6:12] = r1, r2, A3, A4, e1, e2 of the fp64 literal replay.  Computed with NumPy so
    the fp64 constants are the very numbers the reference's ``np.sqrt`` / ``np.exp`` produce."""
    Ua, Ca, Cm, Hm = (np.asarray(x, dtype=np.float64) for x in (Ua, Ca, Cm, Hm))
    a = Cm * Ca / Hm
    b = Cm * (Ua + Hm) / Hm + Ca
    c = Ua
    root = np.sqrt(b * b - 4 * a * c)
    r1 = (-b + root) / (2 * a)
    r2 = (-b - root) / (2 * a)
    A3 = r1 * Ca / Hm + (Ua + Hm) / Hm
    A4 = r2 * Ca / Hm + (Ua + Hm) / Hm
    e1 = np.exp(r1 * dt)
    e2 = np.exp(r2 * dt)

    def F(ta, tm, od, Qa):  # the linear map (Ta, Tm, Tod, Qa) -> (Ta', Tm') on a basis vector
        d = Qa + Ua * od
        dT = Hm * tm / Ca - (Ua + Hm) * ta / Ca + Ua * od / Ca + Qa / Ca
        A1 = (r2 * ta - dT - r2 * d / c) / (r2 - r1)
        A2 = ta - d / c - A1
        return A1 * e1 + A2 * e2 + d / c, A1 * A3 * e1 + A2 * A4 * e2 + d / c

    out = np.empty(Ua.shape + (12,), dtype=np.float64)
    out[..., 0], _ = F(0.0, 1.0, 0.0, 0.0)
    out[..., 1], out[..., 4] = F(0.0, 0.0, 1.0, 0.0)
    out[..., 2], out[..., 5] = F(0.0, 0.0, 0.0, 1.0)
    _, out[..., 3] = F(1.0, 0.0, 0.0, 0.0)
    for k, v in enumerate((r1, r2, A3, A4, e1, e2)):
        out[..., 6 + k] = v
    return out


_HOUSE_F64 = ("t_air", "t_mass", "target", "Ua", "Ca", "Cm", "Hm", "cap")
_ENV_F64 = ("od_temp", "signal", "base_power", "power", "solar", "artificial_ratio", "max_power")


class _DevArray:
    """Minimal ``__cuda_array_interface__`` carrier for zero-copy torch views."""

    def __init__(self, ptr: int, shape, typestr: str, strides=None):
        self.__cuda_array_interface__ = {
            "shape": tuple(int(s) for s in shape), "typestr": typestr, "data": (int(ptr), False),
            "version": 3, "strides": None if strides is None else tuple(int(s) for s in strides),
        }


class DrSim:
    """Owns one ``drsim_t``: R replicas x N houses on one CUDA device."""

    def __init__(self, cfg: _lib.Config, device: int = 0):
        self._L = _lib.lib()
        self.cfg = cfg
        self.device = int(device)
        self._h = C.c_void_p()
        _lib.check(self._L.drsim_create(C.byref(cfg), self.device, C.byref(self._h)))
        self._bind()

    def _bind(self):
        ptrs = _lib.Ptrs()
        _lib.check(self._L.drsim_buffers(self._h, C.byref(ptrs)))
        self.ptrs = ptrs
        self.R, self.N, self.Ns, self.D = ptrs.n_rep, ptrs.n_house, ptrs.house_stride, ptrs.obs_dim
        self.real = np.float64 if ptrs.real_bytes == 8 else np.float32
        self.obs_bf16 = ptrs.obs_bytes == 2   # rows of bfloat16: raw uint16 bits on the numpy side
        self._views: Optional[Dict[str, Any]] = None

    # ---- lifetime -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.drsim_destroy(self._h)
            self._h = C.c_void_p()
            self._views = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def clone(self) -> "DrSim":
        other = object.__new__(DrSim)
        other._L, other.cfg, other.device = self._L, self.cfg, self.device
        other._h = C.c_void_p()
        _lib.check(self._L.drsim_clone(self._h, C.byref(other._h)))
        other._bind()
        return other

    # ---- stream plumbing ------------------------------------------------------------------
    def _stream(self, stream=None) -> C.c_void_p:
        if stream is not None:
            return C.c_void_p(int(getattr(stream, "cuda_stream", stream)))
        import torch

        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- state I/O (host fp64 arrays) -----------------------------------------------------
    def set_state(self, st: Dict[str, Any], stream=None) -> None:
        R, N = self.R, self.N
        hs = _lib.HostState()
        keep = []

        def put(name, arr, dtype, shape, ptype):
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(arr).astype(dtype, copy=False), shape))
            keep.append(a)
            setattr(hs, name, a.ctypes.data_as(ptype))

        for k in _HOUSE_F64:
            if k in st:
                put(k, st[k], np.float64, (R, N), _lib._pd)
        for k in ("on", "lockout"):
            if k in st:
                put(k, np.asarray(st[k]).astype(bool), np.uint8, (R, N), _lib._pu8)
        if "sso" in st:
            put("sso", st["sso"], np.int32, (R, N), _lib._pi32)
        if "lockout_duration" in st:   # per-HVAC durations (legacy lockout_noise): general path only
            put("lockout_duration", st["lockout_duration"], np.int32, (R, N), _lib._pi32)
        if "epoch" in st:
            put("epoch", st["epoch"], np.int64, (R,), _lib._pi64)
        for k in _ENV_F64:
            if k in st:
                put(k, st[k], np.float64, (R,), _lib._pd)
        if "t_since_interp" in st:
            put("t_since_interp", st["t_since_interp"], np.int32, (R,), _lib._pi32)
        if all(k in st for k in ("Ua", "Ca", "Cm", "Hm")):
            bc = lambda k: np.broadcast_to(np.asarray(st[k], dtype=np.float64), (R, N))
            co = thermal_coefs(bc("Ua"), bc("Ca"), bc("Cm"), bc("Hm"), int(self.cfg.dt))
            put("thermal_coefs", co, np.float64, (R, N, 12), _lib._pd)
        _lib.check(self._L.drsim_set_state(self._h, C.byref(hs), self._stream(stream)))

    def get_state(self, keys=None, stream=None) -> Dict[str, np.ndarray]:
        R, N = self.R, self.N
        hs = _lib.HostState()
        out: Dict[str, np.ndarray] = {}
        want = set(keys) if keys else {"t_air", "t_mass", "target", "cap", "on", "lockout", "sso", "epoch",
                                       "od_temp", "signal", "base_power", "power", "solar", "artificial_ratio",
                                       "max_power", "t_since_interp"}

        def get(name, dtype, shape, ptype):
            a = np.zeros(shape, dtype=dtype)
            out[name] = a
            setattr(hs, name, a.ctypes.data_as(ptype))

        for k in ("t_air", "t_mass", "target", "cap"):
            if k in want:
                get(k, np.float64, (R, N), _lib._pd)
        for k in ("on", "lockout"):
            if k in want:
                get(k, np.uint8, (R, N), _lib._pu8)
        if "sso" in want:
            get("sso", np.int32, (R, N), _lib._pi32)
        if "lockout_duration" in want:
            get("lockout_duration", np.int32, (R, N), _lib._pi32)
        if "epoch" in want:
            get("epoch", np.int64, (R,), _lib._pi64)
        for k in _ENV_F64:
            if k in want:
                get(k, np.float64, (R,), _lib._pd)
        if "t_since_interp" in want:
            get("t_since_interp", np.int32, (R,), _lib._pi32)
        _lib.check(self._L.drsim_get_state(self._h, C.byref(hs), self._stream(stream)))
        return out

    def reset_device(self, props, seed: int, mode: str = "reference", quirk_ua: bool = True, stream=None) -> None:
        """``drsim_reset``: draw every house property / initial state on the device from Philox
        streams (the reference's distributions, SURVEY 8a-15).  ``mode``: "reference" (Environment.reset
        semantics incl. quirks Q1-Q3) or "synthetic" (benchmark state of SURVEY 8d)."""
        p = as_props(props)
        hp = p.cluster_prop.house_prop
        a = _lib.ResetArgs()
        a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        a.mode = {"reference": 0, "synthetic": 1}[mode]
        a.randomize_date = int(p.start_datetime_mode == "random")
        a.start_epoch = to_epoch(p.start_datetime)
        a.init_air_temp, a.init_mass_temp = hp.init_air_temp, hp.init_mass_temp
        a.std_target_temp = hp.noise_prop.std_target_temp
        a.factor_low, a.factor_high = hp.noise_prop.factor_thermo_low, hp.noise_prop.factor_thermo_high
        a.quirk_ua = int(quirk_ua)
        caps = list(hp.hvac_prop.noise_prop.cooling_capacity_list)[:8]
        a.n_caps = len(caps)
        for i, c in enumerate(caps):
            a.caps[i] = float(c)
        _lib.check(self._L.drsim_reset(self._h, C.byref(a), self._stream(stream)))

    def set_comm_table(self, table: np.ndarray, stream=None) -> None:
        t = np.ascontiguousarray(np.asarray(table, dtype=np.int32))
        per_rep = 1 if t.ndim == 3 else 0
        want = ((self.R,) if per_rep else ()) + (self.N, self.ptrs.nb_comm)
        if t.shape != want:
            raise ValueError(f"neighbour table shape {t.shape}, expected {want}")
        _lib.check(self._L.drsim_set_comm_table(self._h, t.ctypes.data_as(C.c_void_p), per_rep, self._stream(stream)))

    def set_interp_table(self, table10d: np.ndarray, stream=None) -> None:
        """``table10d``: the flat / 10-D table in the reference's key order
        (``interp_dict_keys.csv``); it is re-ordered here to [162][9][5][8][12][6]."""
        t = np.asarray(table10d, dtype=np.float64).reshape(3, 3, 3, 3, 9, 5, 8, 2, 12, 6)
        t = np.ascontiguousarray(np.moveaxis(t, 7, 4)).reshape(-1)
        _lib.check(self._L.drsim_set_interp_table(self._h, t.ctypes.data_as(C.c_void_p), self._stream(stream)))

    # ---- stepping -------------------------------------------------------------------------
    @staticmethod
    def _ptr(x) -> Optional[int]:
        if x is None:
            return None
        return int(x.data_ptr()) if hasattr(x, "data_ptr") else int(x)

    def _args(self, actions=None, od_noise=None, perlin=None, interp_ids=None) -> _lib.StepArgs:
        a = _lib.StepArgs()
        a.actions, a.od_noise = self._ptr(actions), self._ptr(od_noise)
        a.perlin, a.interp_ids = self._ptr(perlin), self._ptr(interp_ids)
        return a

    def step(self, actions=None, od_noise=None, perlin=None, interp_ids=None, stream=None) -> None:
        """All arguments are device tensors / pointers laid out as ``drsim_step_args`` wants
        (``actions`` u8 with row stride ``Ns``; fp64 noise; int32 ids)."""
        a = self._args(actions, od_noise, perlin, interp_ids)
        _lib.check(self._L.drsim_step(self._h, C.byref(a), self._stream(stream)))

    def run(self, n_steps: int, action_tape=None, stream=None, rotate: bool = False) -> None:
        """``drsim_run`` / ``drsim_run_tape``: ``n_steps`` steps in one call.  ``action_tape``: u8 CUDA tensor
        ``[T, R, Ns]`` (one plane per step; ``rotate=True``: step k reads plane ``k % T``), ``[R, Ns]`` (the same
        plane every step) or None (internal plane / on-device policy)."""
        stride, planes = 0, 0
        if action_tape is not None:
            assert action_tape.is_contiguous() and tuple(action_tape.shape[-2:]) == (self.R, self.Ns)
            if action_tape.dim() == 3:
                assert rotate or action_tape.shape[0] >= n_steps
                stride = self.R * self.Ns
                planes = int(action_tape.shape[0]) if rotate else 0
        a = self._args(action_tape)
        _lib.check(self._L.drsim_run_tape(self._h, C.byref(a), int(n_steps), stride, planes, self._stream(stream)))

    def refresh(self, recompute_signal: bool, od_noise=None, perlin=None, interp_ids=None, stream=None) -> None:
        a = self._args(None, od_noise, perlin, interp_ids)
        _lib.check(self._L.drsim_refresh(self._h, C.byref(a), int(recompute_signal), self._stream(stream)))

    def step_begin(self, actions=None, od_noise=None, perlin=None, interp_ids=None, stream=None) -> None:
        a = self._args(actions, od_noise, perlin, interp_ids)
        _lib.check(self._L.drsim_step_begin(self._h, C.byref(a), self._stream(stream)))

    def step_finish(self, acc=None, n_parts: int = 1, stream=None) -> None:
        """``acc``: gathered per-rank partials ``[n_parts, R, N_ACC]`` (device fp64) or None."""
        a = self._args()
        _lib.check(self._L.drsim_step_finish(self._h, C.byref(a), self._ptr(acc), int(n_parts), self._stream(stream)))

    def step_sharded(self, actions=None, stream=None) -> None:
        """``drsim_step_sharded``: both halves of a house-sharded step in one call (peer exchange / one rank)."""
        a = self._args(actions)
        _lib.check(self._L.drsim_step_sharded(self._h, C.byref(a), self._stream(stream)))

    def step_finish_gathered(self, acc, halo, n_parts: int, rank: int, stream=None) -> None:
        """Gathered partials ``[n_parts, R, N_ACC]`` + gathered halo records
        ``[n_parts, R, nb_comm, HALO_FIELDS]`` (or None when no halo is exchanged), rank order."""
        _lib.check(self._L.drsim_step_finish_gathered(self._h, self._ptr(acc), self._ptr(halo), int(n_parts), int(rank),
                                                      self._stream(stream)))

    def ipc_export(self) -> bytes:
        buf = C.create_string_buffer(96)
        _lib.check(self._L.drsim_ipc_export(self._h, buf))
        return buf.raw

    def ipc_attach(self, rank: int, world: int, handles: list, stream=None) -> None:
        blob = b"".join(handles)
        assert len(blob) == 96 * world
        _lib.check(self._L.drsim_ipc_attach(self._h, int(rank), int(world), blob, self._stream(stream)))

    def peer_status(self, stream=None) -> None:
        _lib.check(self._L.drsim_peer_status(self._h, self._stream(stream)))

    @staticmethod
    def peer_attach_local(sims: list, stream=None) -> None:
        """``drsim_peer_attach_local``: the peer exchange between handles of THIS process, in rank order (raw
        device pointers instead of IPC handles).  Shards that share a GPU must be stepped on different streams."""
        arr = (C.c_void_p * len(sims))(*[s._h for s in sims])
        _lib.check(sims[0]._L.drsim_peer_attach_local(arr, len(sims), sims[0]._stream(stream)))

    def _host_buf(self, x, dtype, shape, keep: list, what: str, writable: bool = False):
        """Pointer of a host buffer handed to the C ABI, after checking what the ABI cannot: dtype, shape and
        contiguity (a wrong stride or a 4-byte dtype would be read as garbage actions)."""
        if x is None:
            return None
        if type(x) is np.ndarray and x.dtype == dtype and x.shape == tuple(shape) and x.flags.c_contiguous:
            keep.append(x)           # already what the ABI wants: no conversion
            return C.c_void_p(x.__array_interface__["data"][0])
        if hasattr(x, "data_ptr"):   # torch CPU tensor (pinned or pageable)
            import torch

            want = {np.uint8: (torch.uint8, torch.bool), np.float64: (torch.float64,), np.float32: (torch.float32,),
                    np.int32: (torch.int32,), np.uint16: (torch.bfloat16,)}[dtype]
            if x.is_cuda or x.dtype not in want or not x.is_contiguous() or tuple(x.shape) != tuple(shape):
                raise ValueError(f"{what}: expected a contiguous CPU tensor of dtype {want[0]} and shape {tuple(shape)}, "
                                 f"got {x.dtype} {tuple(x.shape)} (cuda={x.is_cuda}, contiguous={x.is_contiguous()})")
            return C.c_void_p(x.data_ptr())
        if writable:
            if not (isinstance(x, np.ndarray) and x.dtype == dtype and x.flags.c_contiguous and x.shape == tuple(shape)):
                raise ValueError(f"{what}: expected a C-contiguous numpy array of dtype {np.dtype(dtype)} and shape {tuple(shape)}")
            keep.append(x)
            return x.ctypes.data_as(C.c_void_p)
        a = np.asarray(x)
        if dtype == np.uint8 and a.dtype == np.bool_:
            a = a.view(np.uint8)
        if a.shape != tuple(shape):
            raise ValueError(f"{what}: expected shape {tuple(shape)}, got {a.shape}")
        a = np.ascontiguousarray(a, dtype=dtype)
        keep.append(a)
        return a.ctypes.data_as(C.c_void_p)

    def step_host(self, actions: Optional[np.ndarray], od_noise=None, perlin=None, interp_ids=None,
                  env_out: Optional[np.ndarray] = None, reward_out=None, obs_out=None, stream=None) -> Optional[np.ndarray]:
        """Host-buffer step (``drsim_step_host``): numpy (or pinned torch CPU) buffers in and out.
        ``actions`` uint8 / bool ``[R, N]`` with values 0 / 1; ``env_out`` fp64 ``[R, 4]``.  With ``reward_out``
        ``[R, N]`` and / or ``obs_out`` ``[R, N, D]`` (dtype of the build; with bfloat16 rows a pinned CPU
        ``torch.bfloat16`` tensor or a numpy ``uint16`` array of the raw bits) the call is ``drsim_step_host_full``:
        the reference's full ``step`` result comes back to the host."""
        keep: list = []
        R, N = self.R, self.N
        if env_out is None:
            env_out = np.zeros((R, 4), dtype=np.float64)
        k = int(self.cfg.interp_nb_agents)
        args = [self._host_buf(actions, np.uint8, (R, N), keep, "actions"),
                self._host_buf(None if od_noise is None else np.reshape(od_noise, (R,)), np.float64, (R,), keep, "od_noise"),
                self._host_buf(None if perlin is None else np.reshape(perlin, (R,)), np.float64, (R,), keep, "perlin"),
                self._host_buf(None if interp_ids is None else np.reshape(interp_ids, (R, k)), np.int32, (R, k), keep, "interp_ids"),
                self._host_buf(env_out, np.float64, (R, 4), keep, "env_out", writable=True)]
        if reward_out is None and obs_out is None:
            _lib.check(self._L.drsim_step_host(self._h, *args, self._stream(stream)))
        else:
            args += [self._host_buf(reward_out, self.real, (R, N), keep, "reward_out", writable=True),
                     self._host_buf(obs_out, np.uint16 if self.obs_bf16 else self.real, (R, N, self.D), keep, "obs_out",
                                    writable=True)]
            _lib.check(self._L.drsim_step_host_full(self._h, *args, self._stream(stream)))
        return env_out

    def _snapshot_arrays(self, v: "_lib.SnapshotView") -> Dict[str, np.ndarray]:
        """numpy views of the handle's pinned snapshot (valid until the next snapshot of this handle)."""
        key = (C.cast(v.t_air, C.c_void_p).value, C.cast(v.env, C.c_void_p).value)
        if getattr(self, "_snap_key", None) == key:      # the pinned buffers do not move: reuse the views
            return self._snap_arrays
        R, N, D = self.R, self.N, self.D
        as_arr = np.ctypeslib.as_array
        out = {"t_air": as_arr(v.t_air, (R, N)), "t_mass": as_arr(v.t_mass, (R, N)), "reward": as_arr(v.reward, (R, N)),
               "sso": as_arr(v.sso, (R, N)), "on": as_arr(v.on, (R, N)), "lockout": as_arr(v.lockout, (R, N)),
               "env": as_arr(v.env, (R, 8)), "obs": None}
        if D and v.obs:
            ct = C.c_uint16 if self.obs_bf16 else (C.c_double if self.ptrs.real_bytes == 8 else C.c_float)
            out["obs"] = as_arr(C.cast(v.obs, C.POINTER(ct)), (R, N, D))
        self._snap_key, self._snap_arrays = key, out
        return out

    def snapshot(self, stream=None) -> Dict[str, np.ndarray]:
        """``drsim_snapshot``: what the dict API is built from (absolute temperatures, rewards, seconds_since_off,
        flags, env scalars ``[R, 8]`` = od_temp, signal, power, solar, base_power, epoch, t_since_interp, max_power,
        observation rows) in ONE call / one synchronisation, as numpy views of pinned host memory."""
        v = _lib.SnapshotView()
        _lib.check(self._L.drsim_snapshot(self._h, C.byref(v), self._stream(stream)))
        return self._snapshot_arrays(v)

    def step_host_snapshot(self, actions, od_noise=None, perlin=None, interp_ids=None, stream=None) -> Dict[str, np.ndarray]:
        """``drsim_step_host_snapshot``: the host-buffer step followed by the snapshot, one synchronisation."""
        keep: list = []
        R, N = self.R, self.N
        k = int(self.cfg.interp_nb_agents)
        args = [self._host_buf(actions, np.uint8, (R, N), keep, "actions"),
                self._host_buf(None if od_noise is None else np.reshape(od_noise, (R,)), np.float64, (R,), keep, "od_noise"),
                self._host_buf(None if perlin is None else np.reshape(perlin, (R,)), np.float64, (R,), keep, "perlin"),
                self._host_buf(None if interp_ids is None else np.reshape(interp_ids, (R, k)), np.int32, (R, k), keep, "interp_ids")]
        v = _lib.SnapshotView()
        _lib.check(self._L.drsim_step_host_snapshot(self._h, *args, C.byref(v), self._stream(stream)))
        return self._snapshot_arrays(v)

    ACTOR_PRECISION = {"tf32": 0, "tf32x3": 1}

    def actor_net(self, weights, precision: str = "tf32x3") -> "_lib.ActorNet":
        w1, b1, w2, b2, w3, b3 = weights
        net = _lib.ActorNet()
        net.w1, net.b1, net.w2, net.b2, net.w3, net.b3 = (self._ptr(t) for t in (w1, b1, w2, b2, w3, b3))
        net.h1, net.h2 = int(w1.shape[0]), int(w2.shape[0])
        net.precision = self.ACTOR_PRECISION[precision]
        return net

    def policy_step(self, weights, seed: int = 0, prob_drawn=None, prob_on=None, stream=None, precision: str = "tf32x3") -> None:
        """``drsim_policy_step``: the reference's MA-PPO actor + categorical draw on the observation rows.
        ``weights`` = (w1, b1, w2, b2, w3, b3) contiguous fp32 CUDA tensors in ``torch.nn.Linear`` layout;
        ``prob_drawn`` / ``prob_on``: optional fp32 CUDA tensors ``[R, Ns]``; ``precision``: "tf32x3" (three
        tensor-core passes per product on hi / lo operand halves: fp32-grade probabilities) or "tf32" (one pass)."""
        w1, b1, w2, b2, w3, b3 = weights
        net = self.actor_net(weights, precision)
        assert tuple(w1.shape) == (net.h1, self.D) and tuple(w2.shape) == (net.h2, net.h1) and tuple(w3.shape) == (2, net.h2)
        _lib.check(self._L.drsim_policy_step(self._h, C.byref(net), int(seed) & (2 ** 64 - 1), self._ptr(prob_drawn),
                                             self._ptr(prob_on), self._stream(stream)))

    @property
    def launch_count(self) -> int:
        return int(self._L.drsim_launch_count(self._h))

    @property
    def step_count(self) -> int:
        """Steps taken since creation or the last device reset (``drsim_step_count``)."""
        return int(self._L.drsim_step_count(self._h))

    def comm_sample(self, draw: Optional[int] = None, out=None, stream=None):
        """``random_sample`` handle (``COMM_SAMPLE``): the neighbour table of draw ``draw`` -- default the draw behind
        the current observation rows, i.e. :attr:`step_count` -- as an int32 CUDA tensor ``[R, N, nb_comm]``
        (``drsim_comm_sample``)."""
        import torch

        c = int(self.ptrs.nb_comm)
        if out is None:
            out = torch.empty((self.R, self.N, c), dtype=torch.int32, device=f"cuda:{self.device}")
        assert out.dtype == torch.int32 and out.is_contiguous() and out.numel() == self.R * self.N * c
        _lib.check(self._L.drsim_comm_sample(self._h, -1 if draw is None else int(draw), self._ptr(out), self._stream(stream)))
        return out

    def fused_info(self) -> Dict[str, int]:
        """Geometry of the fused step kernel chosen for this handle (``drsim_fused_info``)."""
        out = (C.c_int32 * 6)()
        _lib.check(self._L.drsim_fused_info(self._h, C.byref(out)))
        names = ("none", "chunked", "direct", "staged", "staged_rows")
        return {"variant": names[out[0]], "envs_per_tile": out[1], "tiles": out[2], "grid": out[3],
                "smem_bytes": out[4], "ctas_per_sm": out[5]}

    @property
    def last_route(self) -> str:
        """Kernels of the last step launched on this handle (``drsim_step_route``; "none" before the first)."""
        names = ("four-kernel", "k_shard", "k_fused", "k_fused_direct", "k_fused_tma<0>", "k_fused_tma<1>", "k_fused_tma<2>",
                 "k_fused_rows<staged>", "k_fused_rows<unstaged>", "k_small", "k_small_gen")
        r = self._L.drsim_step_route(self._h)
        return "none" if r < 0 else names[r]

    def cluster_summary(self, out=None, stream=None):
        """``drsim_cluster_summary``: fp64 CUDA tensor ``[R, 8]`` = locked HVACs, sum Ta, sum (Ta - target),
        sum |Ta - target|, sum Tm, sum target, running HVACs, N  (the UI feed's aggregates,
        client_manager_service.py:64-118,178-197)."""
        import torch

        if out is None:
            out = torch.empty((self.R, _lib.SUMMARY_FIELDS), dtype=torch.float64, device=f"cuda:{self.device}")
        assert out.dtype == torch.float64 and out.is_contiguous() and out.numel() == self.R * _lib.SUMMARY_FIELDS
        _lib.check(self._L.drsim_cluster_summary(self._h, self._ptr(out), self._stream(stream)))
        return out

    # ---- zero-copy torch views ------------------------------------------------------------
    def views(self) -> Dict[str, Any]:
        """Torch CUDA tensors aliasing the library's buffers (no copies).  House planes are
        ``[R, N]`` views of ``[R, Ns]`` storage; ``obs`` is ``[R, N, D]`` (``torch.bfloat16`` on a handle with
        bfloat16 rows)."""
        if self._views is not None:
            return self._views
        import torch

        p, R, N, Ns, D = self.ptrs, self.R, self.N, self.Ns, self.D
        rt = "<f8" if p.real_bytes == 8 else "<f4"
        dev = torch.device("cuda", self.device)

        def t(ptr, shape, typestr):
            if not ptr:
                return None
            x = torch.as_tensor(_DevArray(ptr, shape, typestr), device=dev)
            x._drsim_owner = self  # keep the handle alive as long as a view exists
            return x

        v: Dict[str, Any] = {}
        for k in ("target", "cap", "reward"):
            v[k] = t(getattr(p, k), (R, Ns), rt)[:, :N]
        # fp32 build: the planes hold Ta - target / Tm - target; fp64 build: absolute degC
        ta, tm = t(p.t_air, (R, Ns), rt)[:, :N], t(p.t_mass, (R, Ns), rt)[:, :N]
        v["temp_is_deviation"] = bool(p.temp_is_deviation)
        if p.temp_is_deviation:
            v["dt_air"], v["dt_mass"] = ta, tm
        else:
            v["t_air"], v["t_mass"] = ta, tm
        v["sso"] = t(p.sso, (R, Ns), "<i4")[:, :N]
        v["flags"] = t(p.flags, (R, Ns), "|u1")[:, :N]
        v["actions"] = t(p.actions, (R, Ns), "|u1")[:, :N]
        v["actions_padded"] = t(p.actions, (R, Ns), "|u1")
        if not D:
            v["obs_padded"] = None
        elif self.obs_bf16:   # __cuda_array_interface__ has no bfloat16 typestr: alias the bits as int16
            v["obs_padded"] = t(p.obs, (R, Ns, D), "<i2").view(torch.bfloat16)
            v["obs_padded"]._drsim_owner = self
        else:
            v["obs_padded"] = t(p.obs, (R, Ns, D), rt)
        v["obs"] = v["obs_padded"][:, :N, :] if D else None
        v["epoch"] = t(p.epoch, (R,), "<i8")
        for k in ("od_temp", "signal", "base_power", "power", "solar", "pen_sum", "pen_max", "rew_sig"):
            v[k] = t(getattr(p, k), (R,), "<f8")
        v["metrics"] = t(p.metrics, (R, _lib.N_METRICS), "<f8")
        v["acc"] = t(p.acc, (R, _lib.N_ACC), "<f8")
        if p.halo_out:
            v["halo_out"] = t(p.halo_out, (R, int(p.nb_comm), _lib.HALO_FIELDS), "<f8")
        if p.comm_table:
            v["comm_table"] = t(p.comm_table, (N, p.nb_comm), "<i4")
        self._views = v
        return v
