#!/bin/bash
# Round 4 (1 GPU): shared-gene matrix and fluidity probe at C4 and C5, smoke(), the C4 bench line.
set -u
OUT=${1:?usage: bash scripts/r04a.sh OUTPUT_DIR}
mkdir -p "$OUT"
timeout 400 python scripts/probe_shared_genes.py --configs c4,c5 --out "$OUT" > "$OUT/probe_shared_genes.out" 2>&1
echo "probe rc=$?" > "$OUT/steps.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1
echo "smoke rc=$?" >> "$OUT/steps.log"
timeout 200 python bench.py --gpus 1 --steps 20 --warmup 3 --no-cpu-baseline > "$OUT/bench_c4_n1.json" 2> "$OUT/bench_c4_n1.err"
echo "bench rc=$?" >> "$OUT/steps.log"
cat "$OUT/steps.log" "$OUT/probe_shared_genes.out" "$OUT/smoke.log" "$OUT/bench_c4_n1.json"
