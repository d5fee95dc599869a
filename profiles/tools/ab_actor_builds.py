"""A/B of two builds of libdrsim.so on the split-operand actors ("tf32x3", "f16x3"): outputs bit for bit, then times.

Outputs: on bench.py's C4 and C3 rows with fp32 and with bf16 observation rows, a 100 x 100 actor of fixed weights and a
fixed seed, each build runs drsim_policy_step once per precision ("tf32x3", "f16x3", and "tf32" on fp32 rows) and keeps
actions, prob_drawn and prob_on; the two builds must agree bit for bit.
Times: ab_actor_precision.py's arms (the actor alone; one stored transition) in one process per build, the two builds
alternated three times, then bench.py's default line once per build.  The card's name and power limit are queried,
never set.  Each build is loaded with DRSIM_LIB and DRSIM_NO_REBUILD=1, so a library is never rebuilt from the tree.

    python profiles/tools/ab_actor_builds.py PARENT.so NEW.so [--quick] [--no-bench]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ARMS = [(shape, arm, prec) for shape in ("C4", "C3") for arm in ("actor", "rollout") for prec in ("tf32x3", "f16x3")]


def child(dump, quick):
    sys.path.insert(0, HERE)
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    from ab_actor_precision import SHAPES, arm_actor, arm_rollout, make
    from bench import env_prop_for
    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.rollout import RolloutBuffer

    out = {}
    if dump:
        for shape, (R, N, layout) in SHAPES.items():
            for dtype in ("float32", "bfloat16"):
                env = BatchedEnv(env_prop_for(N), R, precision="f32", obs_layout=layout, noise="philox", seed=1234,
                                 obs_dtype=dtype)
                env.reset()
                torch.manual_seed(0)
                fc = torch.nn.ModuleList([torch.nn.Linear(env.sim.D, 100), torch.nn.Linear(100, 100),
                                          torch.nn.Linear(100, 2)]).cuda()
                w = BatchedEnv.actor_weights(fc)
                sim = env.sim
                for prec in ("tf32x3", "f16x3") + (("tf32",) if dtype == "float32" else ()):
                    pd = torch.full((sim.R, sim.Ns), -1.0, dtype=torch.float32, device="cuda")
                    po = torch.full((sim.R, sim.Ns), -1.0, dtype=torch.float32, device="cuda")
                    sim.policy_step(w, seed=0x1234_5678_9abc_def0, prob_drawn=pd, prob_on=po, precision=prec)
                    sim.actor_status()
                    key = f"{shape}_{dtype}_{prec}"
                    out[key + "_actions"] = env._v["actions"].cpu().numpy().copy()
                    out[key + "_prob_drawn"] = pd.cpu().numpy()
                    out[key + "_prob_on"] = po.cpu().numpy()
                del env
                torch.cuda.empty_cache()
        np.savez(dump, **out)
    res = {}
    for shape in SHAPES:
        env, w = make(shape)
        steps = 8 if quick else 200
        buf = RolloutBuffer(env, steps)
        for prec in ("tf32x3", "f16x3"):
            res[f"{shape} actor {prec}"] = arm_actor(env, w, prec, 20 if quick else 500)[0]
            res[f"{shape} rollout {prec}"] = arm_rollout(env, w, prec, steps, buf)
        del env, buf
        torch.cuda.empty_cache()
    print("RESULT " + json.dumps(res))


def run(lib, args, env_extra=None):
    env = dict(os.environ, DRSIM_LIB=os.path.abspath(lib), DRSIM_NO_REBUILD="1", **(env_extra or {}))
    r = subprocess.run([sys.executable, *args], cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise SystemExit(f"{args} with {lib} failed ({r.returncode})")
    return r.stdout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="*", help="PARENT.so NEW.so")
    ap.add_argument("--quick", action="store_true", help="few calls (a smoke run of the script itself)")
    ap.add_argument("--no-bench", action="store_true", help="skip bench.py's default line")
    ap.add_argument("--child", metavar="DUMP", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child is not None:
        return child(args.child, args.quick)
    if len(args.libs) != 2:
        ap.error("two libraries: PARENT.so NEW.so")
    import numpy as np

    names = ("parent", "new")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    print(smi)
    tmp = tempfile.mkdtemp(prefix="ab_actor_builds_")
    times = {n: {k: [] for k in (f"{s} {a} {p}" for s, a, p in ARMS)} for n in names}
    for rep in range(3):
        for name, lib in zip(names, args.libs):
            dump = os.path.join(tmp, f"{name}.npz") if rep == 0 else ""
            out = run(lib, [os.path.abspath(__file__), "--child", dump] + (["--quick"] if args.quick else []))
            res = json.loads(next(l for l in out.splitlines() if l.startswith("RESULT "))[7:])
            for k, v in res.items():
                times[name][k].append(v)
    a, b = (np.load(os.path.join(tmp, f"{n}.npz")) for n in names)
    assert sorted(a.files) == sorted(b.files)
    print(f"outputs: {len(a.files)} arrays (actions, prob_drawn, prob_on of every shape x row dtype x precision)")
    for k in sorted(a.files):
        same = a[k].tobytes() == b[k].tobytes()
        print(f"  {k:34s} {'bit-identical' if same else 'DIFFERENT: max |d| %.3g' % float(np.abs(a[k].astype(np.float64) - b[k]).max())}")
    print(f"{'arm':22s} {'parent us/call (3 runs)':>30s} {'new us/call (3 runs)':>30s} {'new/parent (medians)':>22s}")
    for k in times["parent"]:
        pa, nb = times["parent"][k], times["new"][k]
        print(f"{k:22s} {'  '.join(f'{x:8.2f}' for x in pa):>30s} {'  '.join(f'{x:8.2f}' for x in nb):>30s} "
              f"{np.median(nb) / np.median(pa):22.3f}")
    if not args.no_bench:
        for name, lib in zip(names, args.libs):
            line = run(lib, ["bench.py", "--gpus", "1"]).strip().splitlines()[-1]
            print(f"bench.py --gpus 1 ({name}): {line}")
    bad = [k for k in a.files if a[k].tobytes() != b[k].tobytes()]
    if bad:
        raise SystemExit(f"{len(bad)} output arrays differ between the builds")


if __name__ == "__main__":
    main()
