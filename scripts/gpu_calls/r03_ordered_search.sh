# Round 3: the culled search in caller order as the engine default.  Expects a checkout of the parent commit in ./_parent
# (built here), measures both in the same session: the new GPU tests, smoke, bench --dump-outputs of both (compared
# array for array), alternating headline bench runs, and the brute/culled comparison of scripts/gpu_ordered_search.py.
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"; export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r03_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r03_build.log 2>&1; echo "build rc=$?"
(cd _parent && python -c "import __graft_entry__ as g; g.build()") > $OUT/r03_build_parent.log 2>&1; echo "parent build rc=$?"
python -m pytest -q -x -m gpu tests/test_ordered_search_gpu.py > $OUT/r03_tests_new.log 2>&1; echo "new tests rc=$?"; tail -3 $OUT/r03_tests_new.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r03_smoke.log 2>&1; echo "smoke rc=$?"
python bench.py --no-sweep --no-cpu-baseline --dump-outputs $OUT/r03_dump_branch > $OUT/r03_dump_branch.json 2>$OUT/r03_dump_branch.err; echo "dump branch rc=$?"
(cd _parent && python bench.py --no-sweep --no-cpu-baseline --dump-outputs ../$OUT/r03_dump_parent) > $OUT/r03_dump_parent.json 2>$OUT/r03_dump_parent.err; echo "dump parent rc=$?"
python - <<'PY'
import glob, os, numpy as np
a, b = os.environ["OUT"] + "/r03_dump_parent", os.environ["OUT"] + "/r03_dump_branch"
names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print("dump arrays", len(names), "different:", bad)
PY
for i in 1 2 3; do
  (cd _parent && python bench.py --no-sweep --no-cpu-baseline) > $OUT/r03_ab_parent_$i.json 2>/dev/null
  python bench.py --no-sweep --no-cpu-baseline > $OUT/r03_ab_branch_$i.json 2>/dev/null
done
python - <<'PY'
import json, os
for who in ("parent", "branch"):
    for i in (1, 2, 3):
        try:
            d = json.loads([l for l in open(f"{os.environ['OUT']}/r03_ab_{who}_{i}.json") if l.startswith("{")][-1])
            print(who, i, d.get("ms_per_step"), (d.get("sustained") or {}).get("ms_per_step"), d.get("pairs_per_s") or d.get("value"))
        except Exception as e:
            print(who, i, "failed", e)
PY
python scripts/gpu_ordered_search.py --out $OUT/r03_ordered_search.jsonl > $OUT/r03_ordered_search.log 2>&1; echo "ordered rc=$?"; cat $OUT/r03_ordered_search.log | tail -5
