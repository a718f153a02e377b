#!/bin/bash
# Cost and agreement of the uint16 retrieval database (profiles/r3b_retrieval_u16_cost.txt) and the
# GPU tests of the uint16 retrieval paths on the same box. Usage:
#   bash tools/runs/run_retrieval_u16.sh [OUT_DIR]
# (default: a new temporary directory); the records are written there.
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3b_build.log" 2>&1 || { tail -40 "$OUT/r3b_build.log"; exit 1; }
timeout 900 python -m pytest tests/test_gpu_retrieval_uint16.py tests/test_gpu_retrieval.py -q -m gpu > "$OUT/r3b_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3b_gpu_tests.log"
timeout 600 python tools/retrieval_u16_cost.py > "$OUT/r3b_retrieval_u16_cost.txt"
echo "cost exit $?"
tail -3 "$OUT/r3b_gpu_tests.log"; head -20 "$OUT/r3b_retrieval_u16_cost.txt"
echo "records in $OUT"
