#!/bin/bash
# A/B of the MODE 1 row assembly of k_fused_tma (16-byte, bank-rotated shared stores) against the parent commit's
# library, in ONE GPU session.
#
# Build both libraries first, on any machine with nvcc (the .so files are gitignored but travel with the tree):
#   git worktree add /tmp/drsim_parent <parent commit>
#   (cd /tmp/drsim_parent && DRSIM_LIB=$OLDPWD/build_ab/parent/libdrsim.so python -m marl_demandresponse_b200._build)
#   python -m marl_demandresponse_b200._build                    # this tree -> marl_demandresponse_b200/libdrsim.so
# Arguments: extra arms as name=path/to/libdrsim.so (timed on C4 next to the two builds).
# Output: one summary on stdout, every bench line and output dump under $OUT.
cd "$(dirname "$0")/../.."
OUT=${OUT:-${TMPDIR:-/tmp}/ab_tile_rows}
mkdir -p "$OUT"
ARMS=("parent=build_ab/parent/libdrsim.so" "new=marl_demandresponse_b200/libdrsim.so" "$@")
for a in "${ARMS[@]}"; do
  [ -f "${a#*=}" ] || { echo "missing library ${a#*=} (arm ${a%%=*}): build it first" >&2; exit 2; }
done
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv

bench() {   # bench <arm> <tag> <bench.py args...>
  local name=${1%%=*} lib=${1#*=} tag=$2; shift 2
  DRSIM_LIB=$lib DRSIM_NO_REBUILD=1 python bench.py "$@" > "$OUT/${name}_$tag.json" 2> "$OUT/${name}_$tag.err" \
    || echo "bench failed: $name $tag (see $OUT/${name}_$tag.err)"
}

# C4 device-resident step time, the arms alternated three times
for i in 1 2 3; do
  for a in "${ARMS[@]}"; do
    bench "$a" "c4_$i" --workload c4 --steps 5000 --no-cpu --no-rollout --no-c5 --dump-outputs "$OUT/${a%%=*}_c4_$i"
  done
done
# one full default line per build (per-step launches, rollout, sharded cluster), C3 and C1
for a in "${ARMS[@]:0:2}"; do
  bench "$a" full
  bench "$a" c3 --workload c3 --no-cpu --no-c5 --no-rollout
  bench "$a" c1 --workload c1 --no-cpu --no-c5 --no-rollout
done
# C4 with bfloat16 rows (bench.py times fp32 rows): the in-kernel loop and one launch per step, the builds alternated
for i in 1 2 3; do
  for a in "${ARMS[@]:0:2}"; do
    DRSIM_LIB=${a#*=} DRSIM_NO_REBUILD=1 python - > "$OUT/${a%%=*}_bf16_$i.json" 2> "$OUT/${a%%=*}_bf16_$i.err" <<'PY' \
      || echo "bf16 arm failed: ${a%%=*} $i"
import json, sys
sys.path.insert(0, "profiles/tools")
from ab_obs_dtype import arm_run
print(json.dumps({"run": arm_run("C4", "bfloat16", 2048, False)[0], "launch": arm_run("C4", "bfloat16", 1000, True)[0]}))
PY
  done
done

python - "$OUT" "${ARMS[@]%%=*}" <<'EOF'
import json, os, sys
import numpy as np

out, arms = sys.argv[1], sys.argv[2:]

def line(name, tag):
    try:
        with open(os.path.join(out, f"{name}_{tag}.json")) as f:
            return json.loads(f.readline())
    except (OSError, ValueError):
        return None

def get(d, path):
    for k in path.split("."):
        d = d.get(k) if isinstance(d, dict) else None
    return d

print("C4 ms_per_step (us), 5000 steps, arms alternated:")
c4 = {}
for a in arms:
    v = [1e3 * d["ms_per_step"] for d in (line(a, f"c4_{i}") for i in (1, 2, 3)) if d]
    c4[a] = v
    if v:
        print(f"  {a:8s} " + "  ".join(f"{x:7.2f}" for x in v) +
              f"   min {min(v):.2f} max {max(v):.2f} spread {100 * (max(v) - min(v)) / min(v):.1f} %")
if c4.get("parent") and c4.get("new"):
    print(f"  worst new / best parent = {max(c4['new']) / min(c4['parent']):.3f}")
print("outputs of the last timed step against the parent's (np.array_equal):")
for a in arms[1:]:
    for i in (1, 2, 3):
        res = []
        for k in ("obs", "reward"):
            try:
                x = np.load(os.path.join(out, f"parent_c4_{i}", k + ".npy"))
                y = np.load(os.path.join(out, f"{a}_c4_{i}", k + ".npy"))
                res.append(f"{k} {np.array_equal(x, y)}")
            except OSError as e:
                res.append(f"{k} missing ({e.filename})")
        print(f"  {a} run {i}: " + ", ".join(res))
print("C4 bfloat16 rows, us/step (3 runs):")
for a in arms[:2]:
    runs = []
    for i in (1, 2, 3):
        try:
            with open(os.path.join(out, f"{a}_bf16_{i}.json")) as f:
                runs.append(json.loads(f.readline()))
        except (OSError, ValueError):
            pass
    for k in ("run", "launch"):
        print(f"  {a:8s} {k:7s} " + "  ".join(f"{r[k]:7.2f}" for r in runs))
print("other figures (parent -> new):")
for tag, path, unit in (("full", "ms_per_step", "ms/step C4"),
                        ("full", "roofline.per_step_launch.ms_per_step", "ms/step C4, one launch per step"),
                        ("full", "roofline.frac", "roofline.frac"), ("full", "roofline.traffic_stale", "traffic_stale"),
                        ("full", "rollout.us_per_transition", "rollout us/transition"),
                        ("full", "sharded_cluster.us_per_step", "sharded cluster us/step"),
                        ("c3", "ms_per_step", "ms/step C3"), ("c1", "ms_per_step", "ms/step C1")):
    vals = [get(line(a, tag), path) if line(a, tag) else None for a in arms[:2]]
    print(f"  {unit:34s} " + "  ->  ".join(str(v) for v in vals))
EOF
