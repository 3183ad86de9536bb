# Round 5: the kinematic fit with the assignment loss (KinematicEngine(assign=...), reart_kin_assign).  Expects a checkout
# of the parent commit in ./_parent (built here).  Records the card, builds both, runs the new tests, then the whole GPU
# suite and smoke, the measurement of scripts/gpu_kinematic_assign.py, bench --dump-outputs of both builds compared array
# for array, and two alternating headline bench runs of each.
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"; export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r05_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r05_build.log 2>&1; echo "build rc=$?"
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/r05_build_parent.log 2>&1; echo "parent build rc=$?"
python -m pytest -q -m gpu tests/test_kinematic_assign_gpu.py > $OUT/r05_tests_new.log 2>&1; echo "new tests rc=$?"; tail -15 $OUT/r05_tests_new.log
python -m pytest -q -m gpu tests --ignore=tests/test_kinematic_assign_gpu.py > $OUT/r05_tests_gpu.log 2>&1; echo "gpu tests rc=$?"; tail -5 $OUT/r05_tests_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r05_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $OUT/r05_smoke.log
python scripts/gpu_kinematic_assign.py --out $OUT/r05_kinematic_assign.jsonl > $OUT/r05_kinematic_assign.log 2>&1; echo "assign rc=$?"; tail -4 $OUT/r05_kinematic_assign.log
python bench.py --no-sweep --no-cpu-baseline --dump-outputs $OUT/r05_dump_branch > $OUT/r05_dump_branch.json 2>$OUT/r05_dump_branch.err; echo "dump branch rc=$?"
(cd _parent && python bench.py --no-sweep --no-cpu-baseline --dump-outputs ../$OUT/r05_dump_parent) > $OUT/r05_dump_parent.json 2>$OUT/r05_dump_parent.err; echo "dump parent rc=$?"
python - <<'PY'
import glob, os, numpy as np
a, b = os.environ["OUT"] + "/r05_dump_parent", os.environ["OUT"] + "/r05_dump_branch"
names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print("dump arrays", len(names), "different:", bad)
PY
for i in 1 2; do
  (cd _parent && python bench.py --no-sweep --no-cpu-baseline --sustained-s 3) > $OUT/r05_ab_parent_$i.json 2>/dev/null
  python bench.py --no-sweep --no-cpu-baseline --sustained-s 3 > $OUT/r05_ab_branch_$i.json 2>/dev/null
done
python - <<'PY'
import json, os
for who in ("parent", "branch"):
    for i in (1, 2):
        try:
            d = json.loads([l for l in open(f"{os.environ['OUT']}/r05_ab_{who}_{i}.json") if l.startswith("{")][-1])
            print(who, i, d.get("ms_per_step"), (d.get("sustained") or {}).get("ms_per_step"), d.get("value"))
        except Exception as e:
            print(who, i, "failed", e)
PY
nvidia-smi --query-gpu=name,power.limit,clocks.sm --format=csv,noheader | tee -a $OUT/r05_gpu.txt
