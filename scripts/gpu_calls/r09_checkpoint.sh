# Round 9: engine checkpoints.  Expects a checkout of the parent commit in ./_parent with its library built.  The card, the
# new checkpoint tests, the whole GPU suite, smoke, bench --dump-outputs of both builds compared array for array (step()
# is unchanged, so every array must be equal), then scripts/gpu_checkpoint_timing.py at cfg3_16k.
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"; export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/r09_gpu.txt
python -m pytest -q -m gpu -rs tests/test_engine_checkpoint_gpu.py > $OUT/r09_ckpt_tests.log 2>&1
echo "checkpoint tests rc=$?"; tail -5 $OUT/r09_ckpt_tests.log
python scripts/gpu_checkpoint_timing.py > $OUT/r09_checkpoint_timing.json 2>$OUT/r09_checkpoint_timing.err
echo "timing rc=$?"; cat $OUT/r09_checkpoint_timing.json
python -m pytest -q -m gpu tests > $OUT/r09_pytest_gpu.log 2>&1
echo "gpu suite rc=$?"; tail -3 $OUT/r09_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r09_smoke.log 2>&1; echo "smoke rc=$?"
python bench.py --no-sweep --no-cpu-baseline --sustained-s 0 --dump-outputs $OUT/r09_dump_branch > $OUT/r09_dump_branch.json 2>$OUT/r09_dump_branch.err; echo "dump branch rc=$?"
(cd _parent && python bench.py --no-sweep --no-cpu-baseline --sustained-s 0 --dump-outputs ../$OUT/r09_dump_parent) > $OUT/r09_dump_parent.json 2>$OUT/r09_dump_parent.err; echo "dump parent rc=$?"
python - <<'PY'
import glob, json, os, numpy as np
o = os.environ["OUT"]
a, b = o + "/r09_dump_parent", o + "/r09_dump_branch"
names = sorted(os.path.basename(p) for p in glob.glob(a + "/*.npy"))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
print("dump arrays", len(names), "different:", bad)
for who in ("parent", "branch"):
    d = json.loads([l for l in open(f"{o}/r09_dump_{who}.json") if l.startswith("{")][-1])
    print(who, d.get("ms_per_step"), d.get("final_loss"))
PY
