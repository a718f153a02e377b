#!/bin/bash
# The per-point projection tests and the rest of the GPU suite, smoke(), the bench outputs against
# the parent commit's library (byte for byte), and the cost of the scale-invariant octant reduction
# (profiles/r3c_*). Needs the parent commit's library built beforehand as
# neural_spectral_codec_b200/libnsc_b200_parent.so (`make` in that commit's csrc/, then copied).
# Usage:
#   bash tools/runs/run_octant_fix.sh [OUT_DIR]
# (default: a new temporary directory); the records are written there.
cd "$(dirname "$0")/../.."
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
PARENT=neural_spectral_codec_b200/libnsc_b200_parent.so
[ -f "$PARENT" ] || { echo "missing $PARENT"; exit 1; }
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3c_build.log" 2>&1 || { tail -40 "$OUT/r3c_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r3c_gpu.txt" 2>&1
timeout 900 python -m pytest tests -m gpu -v --durations=25 > "$OUT/r3c_gpu_tests.log" 2>&1
echo "tests exit $?" >> "$OUT/r3c_gpu_tests.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3c_smoke.log" 2>&1
echo "smoke exit $?" >> "$OUT/r3c_smoke.log"
for arm in parent fixed; do
    if [ $arm = parent ]; then export NSC_LIB=$PWD/$PARENT; else unset NSC_LIB; fi
    timeout 600 python bench.py --gpus 1 --steps 3 --warmup 1 --no-cpu --dump-outputs "$OUT/dump_$arm" \
        > "$OUT/r3c_bench_dump_$arm.json" 2> "$OUT/r3c_bench_dump_$arm.err"
    echo "bench $arm exit $?"
done
unset NSC_LIB
{ for f in "$OUT"/dump_parent/*; do cmp "$f" "$OUT/dump_fixed/$(basename "$f")" && echo "identical $(basename "$f")"; done; } \
    > "$OUT/r3c_dump_compare.txt" 2>&1
timeout 1200 python tools/octant_fix_cost.py --base "$PARENT" > "$OUT/r3c_octant_fix_cost.txt" 2>&1
echo "cost exit $?"
timeout 1500 python tools/ab.py --repeats 3 --steps 30 --tag r3c parent:parent fixed: > "$OUT/r3c_bench_ab.txt" 2>&1
echo "ab exit $?"
rm -rf "$OUT/dump_parent" "$OUT/dump_fixed"
tail -4 "$OUT/r3c_gpu_tests.log"; tail -2 "$OUT/r3c_smoke.log"; cat "$OUT/r3c_dump_compare.txt"
tail -12 "$OUT/r3c_octant_fix_cost.txt" | grep -v '^{'; tail -3 "$OUT/r3c_bench_ab.txt"
echo "records in $OUT"
