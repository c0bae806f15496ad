#!/bin/bash
# Round 4 (1 GPU): the whole GPU suite with the shared-gene matrix and fluidity added.
set -u
OUT=${1:?usage: bash scripts/r04c.sh OUTPUT_DIR}
mkdir -p "$OUT"
timeout 560 python -m pytest tests -m gpu -q -p no:cacheprovider > "$OUT/pytest_gpu.log" 2>&1
echo "pytest rc=$?" > "$OUT/steps.log"
cat "$OUT/steps.log"; tail -15 "$OUT/pytest_gpu.log"
