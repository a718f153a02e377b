#!/bin/bash
# Image widths other than 360 (profiles/r3f_*): the GPU tests of the fused kernel of
# csrc/nsc_anywidth.cu and the reference-vector test of the other widths, then its cost against the
# general kernel at 512, 1024, 2048 and 180 columns (tools/anywidth_cost.py). Usage:
#   bash tools/runs/run_anywidth.sh [OUT_DIR]
# (default: a new temporary directory); the records are written there.
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3f_build.log" 2>&1 || { tail -40 "$OUT/r3f_build.log"; exit 1; }
timeout 600 python -m pytest tests/test_gpu_anywidth_fused.py \
  tests/test_gpu_parity.py::test_other_image_widths_against_reference_vectors -q -m gpu > "$OUT/r3f_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3f_gpu_tests.log"
timeout 420 python tools/anywidth_cost.py > "$OUT/r3f_anywidth_cost.txt" 2>&1
echo "cost exit $?"
tail -30 "$OUT/r3f_gpu_tests.log"; grep -v '^{' "$OUT/r3f_anywidth_cost.txt"
echo "records in $OUT"
