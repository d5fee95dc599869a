"""Per-role phase time lines of k_actor3 ("tf32x3" or "f16x3") (CTA 0, first 8 tiles), from the clock64
stamps of DRSIM_ACTOR_DBG=1.  Both precisions stamp the same phases; a chunk is 32 columns of R1 in both.

    DRSIM_ACTOR_DBG=1 python profiles/tools/actor_phases.py [c3|c4] [tf32x3|f16x3]
"""
import ctypes as C, os, sys
os.environ["DRSIM_ACTOR_DBG"] = "1"
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from bench import env_prop_for
from marl_demandresponse_b200 import BatchedEnv
from marl_demandresponse_b200 import _lib
which = sys.argv[1] if len(sys.argv) > 1 else "c4"
precision = sys.argv[2] if len(sys.argv) > 2 else "tf32x3"
R, N, layout = (4096, 100, "hand_engineered") if which == "c3" else (2048, 1000, "tarmac")
env = BatchedEnv(env_prop_for(N), R, obs_layout=layout, noise="philox", seed=1)
env.reset()
torch.manual_seed(0)
D = env.sim.D
fc = torch.nn.ModuleList([torch.nn.Linear(D, 100), torch.nn.Linear(100, 100), torch.nn.Linear(100, 2)]).cuda()
w = BatchedEnv.actor_weights(fc)
for _ in range(4):
    env.policy_step(w, precision=precision)
torch.cuda.synchronize()
L = _lib.lib()
L.drsim_debug_actor_times.restype = C.c_int
L.drsim_debug_actor_times.argtypes = [C.c_void_p, C.c_void_p]
buf = np.zeros((8, 3, 16), dtype=np.uint64)
n = L.drsim_debug_actor_times(env.sim._h, buf.ctypes.data_as(C.c_void_p))
assert n == buf.size, n
t0 = int(buf[0][buf[0] > 0].min())
names = {0: ["start", "a1 arrived", "fetch issued", "bar1 passed", "chunk0", "chunk1", "chunk2", "chunk3", "chunk4"],
         1: ["wait bar2", "bar2 passed", "R2 drained", "tile done"],
         2: ["a1 ready", "GEMM1 issued", "c0 ready", "c1 ready", "c2 ready", "c3 ready", "c4 ready", "GEMM2 committed"]}
print(f"{which} {precision}: clock64 cycles since the first stamp of CTA 0 (producer warp 0 / consumer warp 8 / MMA warp)")
for it in range(8):
    for role, rn in ((0, "prod"), (2, "mma "), (1, "cons")):
        row = buf[it][role]
        items = [f"{names[role][i]} {int(row[i]) - t0}" for i in range(len(names[role])) if row[i] > 0]
        print(f"tile {it} {rn}: " + " | ".join(items))
