#!/bin/bash
# A/B of the dense draw against a parent build, in ONE process tree on one GPU:
#   tools/ab_dense_draw.sh PARENT_LIB [OUT] [WORKLOADS]
# OUT: directory for the logs, JSON lines and output dumps (default: a new temporary directory, printed first)
# PARENT_LIB: libomc.so of the parent commit, built into an untracked directory of the tree
# (e.g. git worktree add /tmp/parent HEAD~1 && make -C /tmp/parent/openmcmc_b200/csrc && cp /tmp/parent/openmcmc_b200/libomc.so ab_parent/).
# Runs: the card's name / power limit / max SM clock; tests/test_gpu_dense_warp.py; the draw alone at p = 48, 56, 63, 64
# (4096 chains; parent and new); the C2 headline (bench.py --no-cpu --no-e2e
# --no-extras) alternating parent / new 3 times each; --dump-outputs of both and their largest relative difference;
# one parent / new pair of every workload in WORKLOADS (default: c1 c3 c4a c4b c5).
set -u
cd "$(dirname "$0")/.."
PARENT=$(realpath "$1")
OUT=${2:-$(mktemp -d -t ab_dense_draw.XXXXXX)}
echo "output: $OUT"
WLS=${3:-c1 c3 c4a c4b c5}
NEW=$(realpath openmcmc_b200/libomc.so)
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"

timeout 900 python -m pytest -q -p no:cacheprovider tests/test_gpu_dense_warp.py > "$OUT/pytest_dense_warp.log" 2>&1
echo "test_gpu_dense_warp rc=$?"; tail -3 "$OUT/pytest_dense_warp.log"

for p in 48 56 63 64; do
  OMC_LIB=$PARENT timeout 300 python tools/perf_dense_draw.py 4096 $p | sed 's/^/parent /'
  OMC_LIB=$NEW timeout 300 python tools/perf_dense_draw.py 4096 $p | sed 's/^/new    /'
done | tee "$OUT/draw_only.txt"

for r in 1 2 3; do
  for side in parent new; do
    lib=$PARENT; [ $side = new ] && lib=$NEW
    OMC_LIB=$lib timeout 900 python bench.py --gpus 1 --no-cpu --no-e2e --no-extras > "$OUT/c2_${side}_$r.json" 2> "$OUT/c2_${side}_$r.err"
    echo "c2 $side run $r rc=$?"
  done
done
for side in parent new; do
  lib=$PARENT; [ $side = new ] && lib=$NEW
  OMC_LIB=$lib timeout 900 python bench.py --gpus 1 --no-cpu --no-e2e --no-extras --steps 5 --warmup 2 \
    --dump-outputs "$OUT/dump_$side" > "$OUT/c2_dump_$side.json" 2> "$OUT/c2_dump_$side.err"
  echo "dump $side rc=$?"
done
for w in $WLS; do
  for side in parent new; do
    lib=$PARENT; [ $side = new ] && lib=$NEW
    OMC_LIB=$lib timeout 900 python bench.py --gpus 1 --no-cpu --no-e2e --no-extras --workload $w > "$OUT/${w}_$side.json" 2> "$OUT/${w}_$side.err"
    echo "$w $side rc=$?"
  done
done

python - "$OUT" <<'PY'
import glob, json, os, sys
import numpy as np
out = sys.argv[1]
def line(f):
    try:
        return [json.loads(l) for l in open(f) if l.startswith("{")][-1]
    except Exception as e:
        return {"error": repr(e)}
def kms(d):
    r = d.get("roofline") or {}
    return r.get("kernel_ms")
for side in ("parent", "new"):
    ds = [line(f) for f in sorted(glob.glob(f"{out}/c2_{side}_[0-9].json"))]
    print("c2", side, "value", [d.get("value") for d in ds], "ms_per_step", [d.get("ms_per_step") for d in ds],
          "draw kernel_ms", [kms(d) for d in ds])
worst = 0.0
for f in sorted(glob.glob(f"{out}/dump_parent/*.npy")):
    a = np.load(f); b = np.load(f.replace("dump_parent", "dump_new"))
    den = np.maximum(np.abs(a), 1e-300)
    m = np.isfinite(a) & np.isfinite(b)
    rel = float(np.max(np.abs(a[m] - b[m]) / np.maximum(np.abs(a[m]), np.abs(b[m]).max() * 1e-12 + 1e-300))) if m.any() else 0.0
    same_nan = bool(np.array_equal(np.isfinite(a), np.isfinite(b)))
    worst = max(worst, rel)
    print("dump", os.path.basename(f), a.shape, "max rel diff %.3e" % rel, "finite pattern equal", same_nan)
print("dump worst rel diff %.3e" % worst)
for f in sorted(glob.glob(f"{out}/c[0-9]*_parent.json")):
    w = os.path.basename(f).rsplit("_", 1)[0]
    a, b = line(f), line(f.replace("_parent", "_new"))
    print(w, "parent", a.get("value"), a.get("unit"), "new", b.get("value"))
PY
