# Round 7: the relaxation fit with the flow loss on the native iteration (RelaxationEngine(native=True, flow_ref=...),
# reart_flow_grad).  PARENT_DIR: a checkout of the parent commit (built here).  Records the card, builds both, runs
# the new tests, then the whole GPU suite and smoke, the measurement of scripts/gpu_relax_flow.py (and its kernel census in
# a separate run), bench --dump-outputs of both builds compared array for array, and two alternating headline bench runs
# of each.
OUT=${1:?usage: $0 OUTPUT_DIR PARENT_DIR}
PARENT=${2:?usage: $0 OUTPUT_DIR PARENT_DIR}
mkdir -p "$OUT"; OUT=$(cd "$OUT" && pwd); export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r07_gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r07_build.log 2>&1; echo "build rc=$?"
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()") > $OUT/r07_build_parent.log 2>&1; echo "parent build rc=$?"
python -m pytest -q -m gpu tests/test_relax_flow_gpu.py > $OUT/r07_tests_new.log 2>&1; echo "new tests rc=$?"; tail -15 $OUT/r07_tests_new.log
python -m pytest -q -m gpu tests --ignore=tests/test_relax_flow_gpu.py > $OUT/r07_tests_gpu.log 2>&1; echo "gpu tests rc=$?"; tail -5 $OUT/r07_tests_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r07_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $OUT/r07_smoke.log
python scripts/gpu_relax_flow.py --out $OUT/r07_relax_flow.jsonl > $OUT/r07_relax_flow.log 2>&1; echo "flow rc=$?"; tail -4 $OUT/r07_relax_flow.log
python scripts/gpu_relax_flow.py --census --out $OUT/r07_relax_flow.jsonl > $OUT/r07_relax_flow_census.log 2>&1; echo "census rc=$?"
python bench.py --no-sweep --no-cpu-baseline --dump-outputs $OUT/r07_dump_branch > $OUT/r07_dump_branch.json 2>$OUT/r07_dump_branch.err; echo "dump branch rc=$?"
(cd "$PARENT" && python bench.py --no-sweep --no-cpu-baseline --dump-outputs $OUT/r07_dump_parent) > $OUT/r07_dump_parent.json 2>$OUT/r07_dump_parent.err; echo "dump parent rc=$?"
python - <<'PY'
import glob, json, os, numpy as np
a, b = os.environ["OUT"] + "/r07_dump_parent", os.environ["OUT"] + "/r07_dump_branch"
names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print("dump arrays", len(names), "different:", bad)
for who in ("parent", "branch"):
    try:
        d = json.loads([l for l in open(f"{os.environ['OUT']}/r07_dump_{who}.json") if l.startswith("{")][-1])
        print(who, "gpu_launches", d.get("gpu_launches"), "step_kernels", d.get("step_kernels"))
    except Exception as e:
        print(who, "no result line", e)
PY
for i in 1 2; do
  (cd "$PARENT" && python bench.py --no-sweep --no-cpu-baseline --sustained-s 3) > $OUT/r07_ab_parent_$i.json 2>/dev/null
  python bench.py --no-sweep --no-cpu-baseline --sustained-s 3 > $OUT/r07_ab_branch_$i.json 2>/dev/null
done
python - <<'PY'
import json, os
for who in ("parent", "branch"):
    for i in (1, 2):
        try:
            d = json.loads([l for l in open(f"{os.environ['OUT']}/r07_ab_{who}_{i}.json") if l.startswith("{")][-1])
            print(who, i, d.get("ms_per_step"), (d.get("sustained") or {}).get("ms_per_step"), d.get("value"))
        except Exception as e:
            print(who, i, "failed", e)
PY
nvidia-smi --query-gpu=name,power.limit,clocks.sm --format=csv,noheader | tee -a $OUT/r07_gpu.txt
