"""Cost of `random_sample` neighbours drawn on the device: neighbour modes A/B/C in ONE process and one GPU session.

Shape: bench.py's C3 (4,096 x 100 houses, hand-engineered rows, c = 10 neighbours, D = 50), same seed and the same
rotating action tape for every mode.  Modes: `neighbours` (the arithmetic ring), `random_fixed` (a static table,
drawn once) and `random_sample` (a fresh draw per row per step).  Arms, alternated three times:
  run      drsim_run_tape over the tape (the in-kernel step loop)
  launch   the same with DRSIM_NO_STREAM=1 (one launch per step)
and, once per repetition, the sampler alone: drsim_comm_sample writing the [R, N, c] table of one draw (k_comm_sample,
one row per thread, no shared memory), to separate the cost of the draw from the cost of drawing inside a step kernel.
Times are CUDA events around the timed steps after a warm-up; the card's name and power limit are queried, never set.
Usage: python profiles/tools/ab_comm_sample.py [--quick]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import env_prop_for  # noqa: E402
from marl_demandresponse_b200 import BatchedEnv  # noqa: E402

R, N, C = 4096, 100, 10
MODES = ("neighbours", "random_fixed", "random_sample")


def make(mode):
    p = env_prop_for(N)
    p["cluster_prop"]["agents_comm_prop"] = {"mode": mode, "max_nb_agents_communication": C}
    env = BatchedEnv(p, R, precision="f32", obs_layout="hand_engineered", noise="philox", seed=1234)
    env.reset()
    return env


def tape(planes=4):
    g = torch.Generator(device="cuda").manual_seed(1234)
    return (torch.rand((planes, R, N), device="cuda", generator=g) < 0.5).to(torch.uint8)


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn(steps)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps   # us per step


def arm(mode, steps, no_stream):
    env = make(mode)
    tp = tape()
    if no_stream:
        os.environ["DRSIM_NO_STREAM"] = "1"   # read per call by drsim_run_tape
    try:
        env.run(64, tp, rotate=True)
        us = timed(lambda k: env.run(k, tp, rotate=True), steps)
    finally:
        os.environ.pop("DRSIM_NO_STREAM", None)
    return us, env


def table_us(calls):
    env = make("random_sample")
    out = env.sim.comm_sample(0)
    for d in range(10):
        env.sim.comm_sample(d, out=out)
    return timed(lambda k: [env.sim.comm_sample(d, out=out) for d in range(k)], calls)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="few steps (a smoke run of the script itself)")
    args = ap.parse_args()
    q = args.quick
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    print(smi)
    print(f"C3 shape: {R} replicas x {N} houses, c = {C}, D = {10 + 4 * C}, hand-engineered rows")
    arms = [("run", 128 if q else 1024, False), ("launch", 64 if q else 1000, True)]
    res = {(a, m): [] for a, _, _ in arms for m in MODES}
    tables = []
    for rep in range(3):
        tables.append(table_us(20 if q else 500))
        for name, steps, no_stream in arms:
            for mode in MODES:
                us, env = arm(mode, steps, no_stream)
                res[(name, mode)].append(us)
                info = env.sim.fused_info()
                if rep == 0:
                    print(f"  {name} {mode}: variant {info['variant']}, {info['envs_per_tile']} clusters per tile, "
                          f"grid {info['grid']}, {info['ctas_per_sm']} CTAs per SM")
                del env
                torch.cuda.empty_cache()
    print(f"{'arm':8s} {'mode':14s} {'us/step (3 runs)':>30s} {'median / random_fixed':>22s}")
    for name, _, _ in arms:
        ref = np.median(res[(name, "random_fixed")])
        for mode in MODES:
            v = res[(name, mode)]
            print(f"{name:8s} {mode:14s} {'  '.join(f'{x:8.2f}' for x in v):>30s} {np.median(v) / ref:22.3f}")
    print(f"drsim_comm_sample, one [{R}, {N}, {C}] table: {'  '.join(f'{x:8.2f}' for x in tables)} us per call")


if __name__ == "__main__":
    main()
