#!/bin/bash
# Host scans at image widths other than 360 (profiles/r3g_*): the GPU tests of the uint16 epilogue of
# csrc/nsc_anywidth.cu and of the host-buffer pipeline at those widths, then their cost against the
# earlier host path (tools/anywidth_stream_cost.py). Usage:
#   bash tools/runs/run_anywidth_stream.sh [OUT_DIR]
# (default: a new temporary directory); the records are written there.
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3g_build.log" 2>&1 || { tail -40 "$OUT/r3g_build.log"; exit 1; }
nvidia-smi -i 0 --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$OUT/r3g_gpu.txt"
timeout 900 python -m pytest tests/test_gpu_anywidth_stream.py tests/test_anywidth_u16_abi.py -q > "$OUT/r3g_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3g_gpu_tests.log"
timeout 900 python tools/anywidth_stream_cost.py > "$OUT/r3g_anywidth_stream_cost.txt" 2>&1
echo "cost exit $?"
tail -30 "$OUT/r3g_gpu_tests.log"; cat "$OUT/r3g_anywidth_stream_cost.txt"
echo "records in $OUT"
