#!/bin/bash
# A/B of the eigenbasis dense draw against the parent commit, in ONE process tree on one GPU:
#   tools/ab_eigen_draw.sh PARENT_TREE [OUT] [WORKLOADS]
# PARENT_TREE: an untracked directory of this tree holding the parent commit with its libomc.so built
#   (git archive HEAD~1 | tar -x -C ab_parent && make -C ab_parent/openmcmc_b200/csrc); the parent runs its own Python.
# OUT: directory for the logs and JSON lines (default: a new temporary directory, printed first).
# Runs: the card's name / power limit / max SM clock; the GPU test suite and smoke(); tools/perf_eigen_draw.py (prep and
# draw alone at C2 size); the C2 headline (bench.py --no-cpu --no-e2e --no-extras) alternating parent / new 3 times each;
# one parent / new pair of every workload in WORKLOADS (default: c1 c3 c4a c4b c5 c5full); 200 + 1000 free-running C2
# sweeps of both compared in distribution (profiles/r09_distribution.py).
set -u
cd "$(dirname "$0")/.."
PARENT=$(realpath "$1")
OUT=$(realpath -m "${2:-$(mktemp -d -t ab_eigen_draw.XXXXXX)}")
echo "output: $OUT"
WLS=${3:-c1 c3 c4a c4b c5 c5full}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"

timeout 1200 python -m pytest -q -p no:cacheprovider -m gpu tests > "$OUT/pytest_gpu.log" 2>&1
echo "pytest rc=$?" | tee -a "$OUT/pytest_gpu.log"; tail -3 "$OUT/pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" >> "$OUT/pytest_gpu.log" 2>&1
echo "smoke rc=$?" | tee -a "$OUT/pytest_gpu.log"

timeout 300 python tools/perf_eigen_draw.py 4096 64 | tee "$OUT/perf_eigen_draw.txt"

bench() {   # side, out-file, args...
  local side=$1 out=$2
  shift 2
  if [ "$side" = parent ]; then
    (cd "$PARENT" && timeout 900 python bench.py --gpus 1 --no-cpu --no-e2e --no-extras "$@") > "$out.json" 2> "$out.err"
  else
    timeout 900 python bench.py --gpus 1 --no-cpu --no-e2e --no-extras "$@" > "$out.json" 2> "$out.err"
  fi
  echo "$(basename "$out") rc=$?"
}
for r in 1 2 3; do
  for side in parent new; do bench $side "$OUT/c2_${side}_$r"; done
done
for w in $WLS; do
  for side in parent new; do bench $side "$OUT/${w}_$side" --workload "$w"; done
done

timeout 900 python profiles/r09_distribution.py run "$PARENT" "$OUT/dist_parent.npz"
timeout 900 python profiles/r09_distribution.py run . "$OUT/dist_new.npz"
python profiles/r09_distribution.py compare "$OUT/dist_parent.npz" "$OUT/dist_new.npz" | tee "$OUT/distribution.txt"

python - "$OUT" <<'PY'
import glob, json, os, sys
out = sys.argv[1]
def line(f):
    try:
        return [json.loads(l) for l in open(f) if l.startswith("{")][-1]
    except Exception as e:
        return {"error": repr(e)}
for side in ("parent", "new"):
    ds = [line(f) for f in sorted(glob.glob(f"{out}/c2_{side}_[0-9].json"))]
    print("c2", side, "value", [d.get("value") for d in ds], "ms_per_step", [d.get("ms_per_step") for d in ds],
          "draw kernel_ms", [(d.get("roofline") or {}).get("kernel_ms") for d in ds], "chains_failed",
          [d.get("chains_failed") for d in ds])
for f in sorted(glob.glob(f"{out}/c[0-9]*_parent.json")):
    w = os.path.basename(f).rsplit("_", 1)[0]
    a, b = line(f), line(f.replace("_parent", "_new"))
    print(w, "parent", a.get("value"), a.get("unit"), "new", b.get("value"))
PY
