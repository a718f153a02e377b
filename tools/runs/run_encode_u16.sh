#!/bin/bash
# Cost of the uint16 epilogue of the encode kernels (profiles/r3a_encode_u16_cost.txt) and the GPU
# tests of the uint16 paths on the same box. Usage: bash tools/runs/run_encode_u16.sh [OUT_DIR]
# (default: a new temporary directory); the records are written there.
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3a_build.log" 2>&1 || { tail -40 "$OUT/r3a_build.log"; exit 1; }
timeout 900 python -m pytest tests/test_gpu_encode_uint16.py -q -m gpu > "$OUT/r3a_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3a_gpu_tests.log"
timeout 600 python tools/encode_u16_cost.py > "$OUT/r3a_encode_u16_cost.txt"
echo "cost exit $?"
tail -3 "$OUT/r3a_gpu_tests.log"; head -10 "$OUT/r3a_encode_u16_cost.txt"
echo "records in $OUT"
