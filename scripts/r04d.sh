#!/bin/bash
# Round 4 (1 GPU): the rest of the GPU suite after r04c's time window (the last test of test_rarefy_paths.py, the
# shared-gene tests), with durations.
set -u
OUT=${1:?usage: bash scripts/r04d.sh OUTPUT_DIR}
mkdir -p "$OUT"
timeout 500 python -m pytest tests/test_rarefy_paths.py::test_straggler_threshold_in_a_child_process \
    tests/test_shared_genes_gpu.py -m gpu -q -p no:cacheprovider --durations=8 > "$OUT/pytest_gpu_rest.log" 2>&1
echo "pytest rc=$?" > "$OUT/steps.log"
cat "$OUT/steps.log"; tail -22 "$OUT/pytest_gpu_rest.log"
