#!/bin/sh
# Round 6 (bilinear forward operator): GPU tests of the feature, smoke, cost profile, bench against the parent.
OUT=${1:?usage: sh scratch/run_r06.sh OUTPUT_DIR}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)
python -m pytest -q -m gpu tests/test_bilinear_operator.py > "$OUT"/r06_bilinear_tests.txt 2>&1; echo "bilinear tests rc $?"
tail -n 30 "$OUT"/r06_bilinear_tests.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT"/r06_smoke.txt 2>&1; echo "smoke rc $?"
tail -n 3 "$OUT"/r06_smoke.txt
python scratch/bilinear_cost.py --out "$OUT"/r06_bilinear_cost.json > "$OUT"/r06_cost.txt 2>&1; echo "cost rc $?"
tail -n 6 "$OUT"/r06_cost.txt
for i in 1 2; do
  python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline > "$OUT"/r06_bench_new_$i.json 2>"$OUT"/r06_bench_new_$i.err; echo "bench new $i rc $?"
  (cd _parent && python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline > "$OUT"/r06_bench_parent_$i.json 2>"$OUT"/r06_bench_parent_$i.err); echo "bench parent $i rc $?"
done
