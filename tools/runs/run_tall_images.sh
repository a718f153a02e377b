#!/bin/bash
# Images of more than 64 rows (profiles/r3d_*): the GPU tests of the tall kernels, their cost at
# 16 / 64 / 128 rows with the register feed at 12 (product), 8 and 4 points per thread (the tall8
# and tall4 builds), and the phase breakdown of the generic (64 rows) and the tall (128 rows) kernel.
# Usage: bash tools/runs/run_tall_images.sh [OUT_DIR] (default: a new temporary directory).
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
CSRC=neural_spectral_codec_b200/csrc
{ python -c "import __graft_entry__ as g; g.build()" &&
  make -C $CSRC -j8 VARIANT=tall4 DEFS=-DNSC_TALL_PTS=4 &&
  make -C $CSRC -j8 VARIANT=tall8 DEFS=-DNSC_TALL_PTS=8 &&
  make -C $CSRC -j8 VARIANT=phase DEFS=-DNSC_PHASE_TIMING; } > "$OUT/r3d_build.log" 2>&1 || { tail -40 "$OUT/r3d_build.log"; exit 1; }
timeout 1200 python -m pytest tests/test_gpu_tall_images.py -q -m gpu > "$OUT/r3d_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3d_gpu_tests.log"
timeout 900 python tools/tall_image_cost.py --variant tall4=neural_spectral_codec_b200/libnsc_b200_tall4.so \
    --variant tall8=neural_spectral_codec_b200/libnsc_b200_tall8.so > "$OUT/r3d_tall_image_cost.txt" 2>&1
echo "cost exit $?"
for rows in 64 128; do
    NSC_LIB=neural_spectral_codec_b200/libnsc_b200_phase.so timeout 600 python tools/phase_timing.py beam128 $rows \
        > "$OUT/r3d_phase_beam128_e$rows.txt" 2>&1
    echo "phase $rows exit $?"
done
tail -3 "$OUT/r3d_gpu_tests.log"; grep -v '^{' "$OUT/r3d_tall_image_cost.txt"; cat "$OUT"/r3d_phase_*.txt
echo "records in $OUT"
