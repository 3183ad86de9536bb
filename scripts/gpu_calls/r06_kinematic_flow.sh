# Round 6: the kinematic fit with the flow loss (KinematicEngine(flow_ref=...), reart_kin_flow).  Expects a checkout of the
# parent commit in ./_parent (built here).  Records the card, builds both, runs the new tests, then the whole GPU suite and
# smoke, the measurement of scripts/gpu_kinematic_flow.py (and its kernel census in a separate run), bench --dump-outputs
# of both builds compared array for array, and two alternating headline bench runs of each.
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"; export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r06_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r06_build.log 2>&1; echo "build rc=$?"
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/r06_build_parent.log 2>&1; echo "parent build rc=$?"
python -m pytest -q -m gpu tests/test_kinematic_flow_gpu.py > $OUT/r06_tests_new.log 2>&1; echo "new tests rc=$?"; tail -15 $OUT/r06_tests_new.log
python -m pytest -q -m gpu tests --ignore=tests/test_kinematic_flow_gpu.py > $OUT/r06_tests_gpu.log 2>&1; echo "gpu tests rc=$?"; tail -5 $OUT/r06_tests_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r06_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $OUT/r06_smoke.log
python scripts/gpu_kinematic_flow.py --out $OUT/r06_kinematic_flow.jsonl > $OUT/r06_kinematic_flow.log 2>&1; echo "flow rc=$?"; tail -4 $OUT/r06_kinematic_flow.log
python scripts/gpu_kinematic_flow.py --census --out $OUT/r06_kinematic_flow.jsonl > $OUT/r06_kinematic_flow_census.log 2>&1; echo "census rc=$?"
python bench.py --no-sweep --no-cpu-baseline --dump-outputs $OUT/r06_dump_branch > $OUT/r06_dump_branch.json 2>$OUT/r06_dump_branch.err; echo "dump branch rc=$?"
(cd _parent && python bench.py --no-sweep --no-cpu-baseline --dump-outputs ../$OUT/r06_dump_parent) > $OUT/r06_dump_parent.json 2>$OUT/r06_dump_parent.err; echo "dump parent rc=$?"
python - <<'PY'
import glob, os, numpy as np
a, b = os.environ["OUT"] + "/r06_dump_parent", os.environ["OUT"] + "/r06_dump_branch"
names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print("dump arrays", len(names), "different:", bad)
PY
for i in 1 2; do
  (cd _parent && python bench.py --no-sweep --no-cpu-baseline --sustained-s 3) > $OUT/r06_ab_parent_$i.json 2>/dev/null
  python bench.py --no-sweep --no-cpu-baseline --sustained-s 3 > $OUT/r06_ab_branch_$i.json 2>/dev/null
done
python - <<'PY'
import json, os
for who in ("parent", "branch"):
    for i in (1, 2):
        try:
            d = json.loads([l for l in open(f"{os.environ['OUT']}/r06_ab_{who}_{i}.json") if l.startswith("{")][-1])
            print(who, i, d.get("ms_per_step"), (d.get("sustained") or {}).get("ms_per_step"), d.get("value"))
        except Exception as e:
            print(who, i, "failed", e)
PY
nvidia-smi --query-gpu=name,power.limit,clocks.sm --format=csv,noheader | tee -a $OUT/r06_gpu.txt
