"""A/B of the observation-row dtype (``obs_dtype`` float32 vs bfloat16) in ONE process and one GPU session.

Workloads are bench.py's C4 (2,048 x 1,000 houses, TarMAC rows, D = 10) and C3 (4,096 x 100 houses, hand-engineered
rows, D = 50), same seeds and the same rotating action tape for both dtypes.  Arms, alternated three times:
  run      drsim_run_tape over the tape (the in-kernel step loop)
  launch   the same with DRSIM_NO_STREAM=1 (one launch per step)
  e2e      C4 drsim_step_host_full: pinned actions in, per-agent rewards and rows out
  rollout  C4 drsim_rollout_transition (3xTF32 actor + step into a device rollout buffer)
Times are CUDA events around the timed steps after a warm-up; the card's name and power limit are queried, never set.
Usage: python profiles/tools/ab_obs_dtype.py [--quick]
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
from marl_demandresponse_b200.rollout import RolloutBuffer  # noqa: E402

SHAPES = {"C4": (2048, 1000, "tarmac"), "C3": (4096, 100, "hand_engineered")}


def make(shape, dtype):
    R, N, layout = SHAPES[shape]
    env = BatchedEnv(env_prop_for(N), R, precision="f32", obs_layout=layout, noise="philox", seed=1234, obs_dtype=dtype)
    env.reset()
    return env


def tape(env, planes=4):
    g = torch.Generator(device="cuda").manual_seed(1234)
    return (torch.rand((planes, env.n_replicas, env.n_houses), device="cuda", generator=g) < 0.5).to(torch.uint8)


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn(steps)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps   # us per step


def arm_run(shape, dtype, steps, no_stream):
    env = make(shape, dtype)
    tp = tape(env)
    if no_stream:
        os.environ["DRSIM_NO_STREAM"] = "1"   # read per call by drsim_run_tape
    try:
        env.run(64, tp, rotate=True)
        us = timed(lambda k: env.run(k, tp, rotate=True), steps)
    finally:
        os.environ.pop("DRSIM_NO_STREAM", None)
    return us, env


def arm_e2e(dtype, steps):
    env = make("C4", dtype)
    R, N, D = env.n_replicas, env.n_houses, env.sim.D
    acts = [torch.from_numpy((np.random.default_rng(i).random((R, N)) < 0.5).astype(np.uint8)).pin_memory() for i in range(4)]
    rew = torch.empty((R, N), dtype=torch.float32).pin_memory()
    obs = torch.empty((R, N, D), dtype=torch.bfloat16 if dtype == "bfloat16" else torch.float32).pin_memory()

    def go(k):
        for t in range(k):
            env.step_host(acts[t % 4], reward_out=rew, obs_out=obs)

    go(10)
    return timed(go, steps), env


def arm_rollout(dtype, steps):
    env = make("C4", dtype)
    g = torch.Generator().manual_seed(5)
    w = []
    for fi, fo in ((env.sim.D, 32), (32, 32), (32, 2)):
        w += [(torch.randn((fo, fi), generator=g) / fi ** 0.5).cuda().contiguous(), torch.zeros(fo).cuda()]
    buf = RolloutBuffer(env, steps)
    env.collect(w, buf, n_steps=4, seed=3)
    return timed(lambda k: env.collect(w, buf, n_steps=k, seed=3), steps), env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="few steps (a smoke run of the script itself)")
    args = ap.parse_args()
    q = args.quick
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    print(smi)
    arms = [("C4 run", lambda d: arm_run("C4", d, 128 if q else 2048, False)),
            ("C4 launch", lambda d: arm_run("C4", d, 64 if q else 1000, True)),
            ("C3 run", lambda d: arm_run("C3", d, 128 if q else 1024, False)),
            ("C3 launch", lambda d: arm_run("C3", d, 64 if q else 1000, True)),
            ("C4 e2e full", lambda d: arm_e2e(d, 5 if q else 60)),
            ("C4 rollout", lambda d: arm_rollout(d, 4 if q else 48))]
    res = {name: {"float32": [], "bfloat16": []} for name, _ in arms}
    for rep in range(3):
        for name, fn in arms:
            envs = {}
            for dtype in ("float32", "bfloat16"):
                us, envs[dtype] = fn(dtype)
                res[name][dtype].append(us)
            a, b = envs["float32"].state["obs_padded"], envs["bfloat16"].state["obs_padded"]
            same = torch.equal(b.view(torch.int16), a.to(torch.bfloat16).view(torch.int16)) and \
                torch.equal(envs["float32"].state["reward"], envs["bfloat16"].state["reward"])
            if not same:
                print(f"  !! {name} rep {rep}: bf16 rows / rewards differ from the fp32 handle's")
            del envs
            torch.cuda.empty_cache()
    print(f"{'arm':12s} {'float32 us/step (3 runs)':>30s} {'bfloat16 us/step (3 runs)':>30s} {'bf16/fp32 (medians)':>20s}")
    for name, _ in arms:
        f, b = res[name]["float32"], res[name]["bfloat16"]
        print(f"{name:12s} {'  '.join(f'{x:8.2f}' for x in f):>30s} {'  '.join(f'{x:8.2f}' for x in b):>30s} "
              f"{np.median(b) / np.median(f):20.3f}")


if __name__ == "__main__":
    main()
