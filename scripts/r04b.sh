#!/bin/bash
# Round 4 (1 GPU): shared-gene GEMM with grouped tile order: its GPU tests, the C4 / C5 probe, smoke().
set -u
OUT=${1:?usage: bash scripts/r04b.sh OUTPUT_DIR}
mkdir -p "$OUT"
timeout 300 python -m pytest tests/test_shared_genes_gpu.py -m gpu -x -q > "$OUT/pytest_shared_gpu.log" 2>&1
echo "pytest rc=$?" > "$OUT/steps.log"
timeout 400 python scripts/probe_shared_genes.py --configs c4,c5 --out "$OUT" > "$OUT/probe_shared_genes.out" 2>&1
echo "probe rc=$?" >> "$OUT/steps.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1
echo "smoke rc=$?" >> "$OUT/steps.log"
cat "$OUT/steps.log"; tail -3 "$OUT/pytest_shared_gpu.log"; grep -v Warn "$OUT/probe_shared_genes.out"; cat "$OUT/smoke.log"
