#!/bin/bash
# Host half of libpgx_b200 (csrc/pgx_rng.cpp, pgx_plan.cpp, pgx_plan_build.cpp, pgx_expand.cpp, pgx_inflate.cpp: threaded C++)
# under AddressSanitizer + UndefinedBehaviorSanitizer, driven by the CPU test suite.  No GPU needed.
#
#   bash scripts/sanitize_host.sh [pytest args]      (default: the plan / ABI / sparse_utils / distributed tests)
#   PGX_SANITIZE=thread bash scripts/sanitize_host.sh   the same under ThreadSanitizer (reports are printed, grep
#                                                        the output for "ThreadSanitizer"; the C4 plan takes 36 s)
#
# The sanitized library is built under /tmp (never in-tree: in-tree .so files travel to the GPU box) and
# selected with PGX_LIBRARY; libasan is preloaded because the python binary itself is not instrumented.
set -eu
REPO=$(cd "$(dirname "$0")/.." && pwd)
MODE=${PGX_SANITIZE:-address}
OUT=${PGX_SANITIZE_DIR:-/tmp/pgx_$MODE}
CSRC=$REPO/pangenomix_b200/csrc
mkdir -p "$OUT"
if [ "$MODE" = thread ]; then
  SAN="-fsanitize=thread -fno-omit-frame-pointer"; LINK=""; PRE="$(gcc -print-file-name=libtsan.so)"
else
  SAN="-fsanitize=address,undefined -fno-omit-frame-pointer -fno-sanitize-recover=undefined"
  LINK="-Xlinker $(gcc -print-file-name=libubsan.so)"
  PRE="$(gcc -print-file-name=libasan.so) $(gcc -print-file-name=libubsan.so)"
fi
for src in pgx_rng pgx_plan pgx_inflate pgx_expand pgx_plan_build; do
  g++ -O1 -g -std=c++17 -fPIC -pthread $SAN -I "$REPO/include" -c "$CSRC/$src.cpp" -o "$OUT/$src.o"
done
nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC,-O3,-pthread -shared \
  -I "$REPO/include" -I "$CSRC" -o "$OUT/libpgx_b200.so" \
  "$CSRC/pgx_api.cu" "$CSRC/pgx_rarefy.cu" "$CSRC/pgx_bernoulli.cu" "$CSRC/pgx_heaps.cu" "$CSRC/pgx_betabin.cu" "$CSRC/pgx_perm.cu" "$OUT/pgx_rng.o" "$OUT/pgx_plan.o" "$OUT/pgx_inflate.o" "$OUT/pgx_expand.o" "$OUT/pgx_plan_build.o" \
  $LINK
cd "$REPO"
if [ $# -eq 0 ]; then set -- tests/test_plan.py tests/test_abi_cpu.py tests/test_sparse_utils.py tests/test_distributed_cpu.py; fi
# reports go to files: pytest captures stderr and a sanitizer exit inside a test would take the report with it
rm -f "$OUT"/report.*
RC=0
LD_PRELOAD="$PRE" TSAN_OPTIONS=halt_on_error=0:report_signal_unsafe=0:log_path="$OUT/report" \
ASAN_OPTIONS=detect_leaks=0:allocator_may_return_null=1:log_path="$OUT/report" \
UBSAN_OPTIONS=print_stacktrace=1:halt_on_error=1:log_path="$OUT/report" \
PGX_LIBRARY="$OUT/libpgx_b200.so" python -m pytest "$@" -x -q -m "not gpu" -p no:cacheprovider || RC=$?
if ls "$OUT"/report.* > /dev/null 2>&1; then
  echo "SANITIZER REPORTS:"; head -n 40 "$OUT"/report.*; exit 1
fi
echo "no sanitizer report"
exit $RC
