# Round 8: the culled search's rows grouped per frame on the posed cloud (reart_skinned_chamfer_fwd_bwd_posed).  Expects a
# checkout of the parent commit in ./_parent with both libraries built.  Part "check": the card, the GPU tests of the
# ordered searches, smoke, bench --dump-outputs of both builds compared array for array.  Part "time": alternating
# headline bench runs, then scripts/gpu_posed_order.py on both (blocks evaluated, tie points, ms/step and per-kernel
# times in the headline window and 600 steps into a fit).
OUT=${1:?usage: $0 OUTPUT_DIR check|time}
mkdir -p "$OUT"; export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r08_gpu_$2.txt
if [ "$2" = check ]; then
python -m pytest -q -x -m gpu tests/test_posed_order_gpu.py tests/test_ordered_search_gpu.py > $OUT/r08_tests.log 2>&1
echo "tests rc=$?"; tail -3 $OUT/r08_tests.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r08_smoke.log 2>&1; echo "smoke rc=$?"
python bench.py --no-sweep --no-cpu-baseline --sustained-s 0 --dump-outputs $OUT/r08_dump_branch > $OUT/r08_dump_branch.json 2>$OUT/r08_dump_branch.err; echo "dump branch rc=$?"
(cd _parent && python bench.py --no-sweep --no-cpu-baseline --sustained-s 0 --dump-outputs ../$OUT/r08_dump_parent) > $OUT/r08_dump_parent.json 2>$OUT/r08_dump_parent.err; echo "dump parent rc=$?"
python - <<'PY'
import glob, os, numpy as np
a, b = os.environ["OUT"] + "/r08_dump_parent", os.environ["OUT"] + "/r08_dump_branch"
names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print("dump arrays", len(names), "different:", bad)
PY
else
for i in 1 2; do
  (cd _parent && python bench.py --no-sweep --no-cpu-baseline) > $OUT/r08_ab_parent_$i.json 2>/dev/null
  python bench.py --no-sweep --no-cpu-baseline > $OUT/r08_ab_branch_$i.json 2>/dev/null
done
python - <<'PY'
import json, os
for who in ("parent", "branch"):
    for i in (1, 2):
        try:
            d = json.loads([l for l in open(f"{os.environ['OUT']}/r08_ab_{who}_{i}.json") if l.startswith("{")][-1])
            print(who, i, d.get("ms_per_step"), (d.get("sustained") or {}).get("ms_per_step"), d.get("final_loss"))
        except Exception as e:
            print(who, i, "failed", e)
PY
cp scripts/gpu_posed_order.py _parent/scripts/                       # the measurement script, run on the parent's package
(cd _parent && python scripts/gpu_posed_order.py --out ../$OUT/r08_stats_parent.jsonl --profile ../$OUT/r08_prof_parent) \
    > $OUT/r08_stats_parent.log 2>&1; echo "stats parent rc=$?"; tail -2 $OUT/r08_stats_parent.log
python scripts/gpu_posed_order.py --out $OUT/r08_stats_branch.jsonl --profile $OUT/r08_prof_branch > $OUT/r08_stats_branch.log 2>&1
echo "stats branch rc=$?"; tail -2 $OUT/r08_stats_branch.log
fi
