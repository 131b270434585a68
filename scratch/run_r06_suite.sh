#!/bin/sh
# Round 6: the whole GPU test suite and smoke() from the final tree.
OUT=${1:?usage: sh scratch/run_r06_suite.sh OUTPUT_DIR}
OUT=$(mkdir -p "$OUT" && cd "$OUT" && pwd)
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT"/r06_final_smoke.txt 2>&1; echo "smoke rc $?"
tail -n 2 "$OUT"/r06_final_smoke.txt
python -m pytest -q -m gpu tests --durations=15 > "$OUT"/r06_gpu_suite.txt 2>&1; echo "gpu suite rc $?"
tail -n 40 "$OUT"/r06_gpu_suite.txt
