"""A/B of the actor precision ("tf32x3" vs "f16x3") in ONE process and one GPU session.

Workloads: bench.py's C4 (2,048 x 1,000 houses, TarMAC rows, D = 10) and C3 (4,096 x 100 houses, hand-engineered rows,
D = 50), each with a 100 x 100 actor (the reference's hidden widths).  Arms, the two precisions alternated three times:
  actor    drsim_policy_step alone on the handle's rows (pack + actor launch)
  rollout  one stored transition, drsim_rollout_transition (actor + env step into a device rollout buffer) via collect
Times are CUDA events around many calls after a warm-up.  The card's name and power limit are queried, never set.  The
f16x3 probabilities are compared with the tf32x3 ones on the same rows (max |dp|).
Usage: python profiles/tools/ab_actor_precision.py [--quick]
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
PRECISIONS = ("tf32x3", "f16x3")


def make(shape):
    R, N, layout = SHAPES[shape]
    env = BatchedEnv(env_prop_for(N), R, precision="f32", obs_layout=layout, noise="philox", seed=1234)
    env.reset()
    torch.manual_seed(0)
    fc = torch.nn.ModuleList([torch.nn.Linear(env.sim.D, 100), torch.nn.Linear(100, 100), torch.nn.Linear(100, 2)]).cuda()
    return env, BatchedEnv.actor_weights(fc)


def timed(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn(calls)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / calls   # us per call


def arm_actor(env, w, prec, calls):
    sim = env.sim
    p_on = torch.zeros((sim.R, sim.Ns), dtype=torch.float32, device="cuda")

    def go(k):
        for _ in range(k):
            sim.policy_step(w, seed=7, prob_on=p_on, precision=prec)

    go(20)
    us = timed(go, calls)
    sim.actor_status()
    return us, p_on.clone()


def arm_rollout(env, w, prec, steps, buf):
    env.collect(w, buf, n_steps=4, seed=3, precision=prec)
    return timed(lambda k: env.collect(w, buf, n_steps=k, seed=3, precision=prec), steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="few calls (a smoke run of the script itself)")
    args = ap.parse_args()
    q = args.quick
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    print(smi)
    res = {}
    for shape in SHAPES:
        env, w = make(shape)
        steps = 8 if q else 200
        buf = RolloutBuffer(env, steps)
        dp = 0.0
        for rep in range(3):
            probs = {}
            for prec in PRECISIONS:
                us, probs[prec] = arm_actor(env, w, prec, 20 if q else 500)
                res.setdefault((shape, "actor"), {}).setdefault(prec, []).append(us)
            dp = max(dp, float((probs["f16x3"] - probs["tf32x3"]).abs().max()))
            for prec in PRECISIONS:
                res.setdefault((shape, "rollout"), {}).setdefault(prec, []).append(arm_rollout(env, w, prec, steps, buf))
        res[(shape, "dp")] = dp
        del env, buf
        torch.cuda.empty_cache()
    print(f"{'arm':12s} {'tf32x3 us/call (3 runs)':>30s} {'f16x3 us/call (3 runs)':>30s} {'f16x3/tf32x3 (medians)':>24s}")
    for shape in SHAPES:
        for arm in ("actor", "rollout"):
            a, b = res[(shape, arm)]["tf32x3"], res[(shape, arm)]["f16x3"]
            print(f"{shape + ' ' + arm:12s} {'  '.join(f'{x:8.2f}' for x in a):>30s} {'  '.join(f'{x:8.2f}' for x in b):>30s} "
                  f"{np.median(b) / np.median(a):24.3f}")
    for shape in SHAPES:
        print(f"{shape}: max |p_on(f16x3) - p_on(tf32x3)| on the same rows {res[(shape, 'dp')]:.3g}")


if __name__ == "__main__":
    main()
