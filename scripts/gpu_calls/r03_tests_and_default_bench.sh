# Round 3: the whole GPU suite, then one default bench (headline + sweep) with the culled search in caller order.
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"; export OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03_gpu2.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r03_build2.log 2>&1; echo "build rc=$?"
python -m pytest -q -m gpu tests > $OUT/r03_tests_gpu.log 2>&1; echo "gpu tests rc=$?"; tail -5 $OUT/r03_tests_gpu.log
python bench.py > $OUT/r03_bench_default.json 2> $OUT/r03_bench_default.err; echo "bench rc=$?"
