#!/bin/bash
# Cost of ranking the whole retrieval database (tools/retrieval_rank_cost.py: the device radix sort
# against the torch path it replaced, and the 8-bit digit build against an 11-bit one) and the GPU
# tests of the rank on the same box. Usage:
#   bash tools/runs/run_retrieval_rank.sh [OUT_DIR]
# (default: a new temporary directory); the records are written there.
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
{ python -c "import __graft_entry__ as g; g.build()" &&
  make -C neural_spectral_codec_b200/csrc -j4 VARIANT=rank11 DEFS=-DNSC_RANK_BITS=11; } > "$OUT/r3e_build.log" 2>&1 ||
  { tail -40 "$OUT/r3e_build.log"; exit 1; }
timeout 900 python -m pytest tests/test_gpu_retrieval_rank.py tests/test_gpu_retrieval.py tests/test_gpu_retrieval_uint16.py \
  -q -m gpu > "$OUT/r3e_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3e_gpu_tests.log"
timeout 1200 python tools/retrieval_rank_cost.py --alt-lib neural_spectral_codec_b200/libnsc_b200_rank11.so \
  > "$OUT/r3e_retrieval_rank_cost.txt"
echo "cost exit $?"
tail -3 "$OUT/r3e_gpu_tests.log"; head -14 "$OUT/r3e_retrieval_rank_cost.txt"
echo "records in $OUT"
