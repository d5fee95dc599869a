"""NumPy restatement of the reference's running metrics -- TEST INFRASTRUCTURE (see oracle/__init__.py).

Follows ``server/app/services/metrics_service.py`` literally, slips included: ``Metrics.update`` :108-157
(``temp_error = indoor_temp - target_temp / nb_agents`` -- the division binds to the set-point only, :131-134;
``signal_error = (reg_signal - cluster_hvac_power) / nb_agents**2`` accumulated once per agent, :143-148),
``update_rms`` :237-257, ``reset`` :222-235.  Pinned on values recorded from the real class
(tests/golden/make_golden_metrics.py -> tests/golden/metrics_*.json).
"""
from __future__ import annotations

import numpy as np

FIELDS = ["cumul_avg_reward", "cumul_temp_offset", "cumul_temp_error", "max_temp_error", "cumul_signal_offset",
          "cumul_signal_error", "cumul_squared_error_temp", "cumul_OD_temp", "cumul_signal", "cumul_cons",
          "cumul_squared_error_sig", "cumul_squared_max_error_temp"]


class RefMetrics:
    def __init__(self, nb_agents: int, start_stats_from: int = 0):
        self.n = int(nb_agents)
        self.start = int(start_stats_from)
        self.v = dict.fromkeys(FIELDS, 0.0)

    def update(self, t_air_next, target, rewards, signal_old, power_new, od_old, power_old, time_step: int) -> None:
        """``t_air_next, target, rewards``: [N] after the step; ``signal_old, od_old, power_old``: the observation
        BEFORE the step (metrics_service.py:150-152 read ``obs_dict[0]``); ``power_new``: cluster power after it."""
        v, n = self.v, self.n
        for k in range(n):                                                     # :130
            temp_error = float(t_air_next[k]) - float(target[k]) / n           # :131-134
            v["cumul_temp_offset"] += temp_error
            v["cumul_temp_error"] += abs(temp_error)
            v["max_temp_error"] = max(v["max_temp_error"], temp_error)
            v["cumul_avg_reward"] += float(rewards[k]) / n
            if time_step >= self.start:
                v["cumul_squared_error_temp"] += temp_error ** 2
            signal_error = (float(signal_old) - float(power_new)) / (n ** 2)   # :143-145
            v["cumul_signal_offset"] += signal_error
            v["cumul_signal_error"] += abs(signal_error)
        v["cumul_OD_temp"] += float(od_old)                                    # :150-152
        v["cumul_signal"] += float(signal_old)
        v["cumul_cons"] += float(power_old)
        if time_step >= self.start:
            v["cumul_squared_error_sig"] += float(signal_old) ** 2
            v["cumul_squared_max_error_temp"] = v["max_temp_error"] ** 2

    def row(self):
        return [self.v[f] for f in FIELDS]

    def rms(self, time_step: int) -> dict:                                     # :237-257
        d = time_step - self.start
        return {"rmse_sig_per_ag": float(np.sqrt(self.v["cumul_squared_error_sig"] / d) / self.n),
                "rmse_temp": float(np.sqrt(self.v["cumul_squared_error_temp"] / (d * self.n))),
                "rms_max_error_temp": float(np.sqrt(self.v["cumul_squared_max_error_temp"] / d))}


# Metrics.reset (:222-235) zeroes these and leaves the squared sums alone
RESET_FIELDS = [f for f in FIELDS if f not in ("cumul_squared_error_temp", "cumul_squared_error_sig",
                                               "cumul_squared_max_error_temp")]


class BatchedRefMetrics:
    """``RefMetrics`` of R clusters at once: the same expressions in the same order of updates, with the per-house
    loop of ``update`` as fp64 sums over the house axis of ``[R, N]`` arrays.  ``values`` is ``[R, 12]`` in the order
    of ``FIELDS``."""

    def __init__(self, n_replicas: int, nb_agents: int, start_stats_from: int = 0):
        self.n = int(nb_agents)
        self.start = int(start_stats_from)
        self.values = np.zeros((int(n_replicas), len(FIELDS)))

    def update(self, t_air_next, target, rewards, signal_old, power_new, od_old, power_old, time_step: int) -> None:
        """``t_air_next, target, rewards``: ``[R, N]`` after the step; ``signal_old, od_old, power_old``: ``[R]``, the
        observation BEFORE the step; ``power_new``: ``[R]``, cluster power after it (see ``RefMetrics.update``)."""
        v, n = self.values, self.n
        ix = FIELDS.index
        temp_error = np.asarray(t_air_next, dtype=np.float64) - np.asarray(target, dtype=np.float64) / n
        v[:, ix("cumul_temp_offset")] += temp_error.sum(axis=1)
        v[:, ix("cumul_temp_error")] += np.abs(temp_error).sum(axis=1)
        v[:, ix("max_temp_error")] = np.maximum(v[:, ix("max_temp_error")], temp_error.max(axis=1))
        v[:, ix("cumul_avg_reward")] += (np.asarray(rewards, dtype=np.float64) / n).sum(axis=1)
        if time_step >= self.start:
            v[:, ix("cumul_squared_error_temp")] += (temp_error ** 2).sum(axis=1)
        signal_error = (np.asarray(signal_old, dtype=np.float64) - np.asarray(power_new, dtype=np.float64)) / (n ** 2)
        v[:, ix("cumul_signal_offset")] += n * signal_error
        v[:, ix("cumul_signal_error")] += n * np.abs(signal_error)
        v[:, ix("cumul_OD_temp")] += od_old
        v[:, ix("cumul_signal")] += signal_old
        v[:, ix("cumul_cons")] += power_old
        if time_step >= self.start:
            v[:, ix("cumul_squared_error_sig")] += np.asarray(signal_old, dtype=np.float64) ** 2
            v[:, ix("cumul_squared_max_error_temp")] = v[:, ix("max_temp_error")] ** 2

    def reset(self) -> None:                                                   # :222-235
        self.values[:, [FIELDS.index(f) for f in RESET_FIELDS]] = 0.0

    def rms(self, time_step: int) -> dict:
        d = time_step - self.start
        v, ix = self.values, FIELDS.index
        return {"rmse_sig_per_ag": np.sqrt(v[:, ix("cumul_squared_error_sig")] / d) / self.n,
                "rmse_temp": np.sqrt(v[:, ix("cumul_squared_error_temp")] / (d * self.n)),
                "rms_max_error_temp": np.sqrt(v[:, ix("cumul_squared_max_error_temp")] / d)}
