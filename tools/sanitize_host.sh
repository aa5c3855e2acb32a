#!/bin/bash
# Runs the CPU test suite's native pieces (BAM decoder + inflate, synthetic-data generator, CPU oracle) under
# AddressSanitizer + UndefinedBehaviorSanitizer: builds sanitized copies of the three host libraries in place, runs
# the tests that load them with the sanitizer runtimes preloaded into python, prints every report, rebuilds the
# normal libraries.  2026-10-22: 224 tests, no report (an earlier run found a qsort(NULL, 0) in the oracle, fixed; never one in the decoder).
set -e
cd "$(dirname "$0")/.."
SAN="-O1 -g -fsanitize=address,undefined -fno-omit-frame-pointer -fPIC -shared -std=c11"
gcc $SAN -o himut_b200/libhimut_io.so himut_b200/csrc/bamdec.c -lz -lpthread
gcc $SAN -o himut_b200/libhimut_synth.so himut_b200/csrc/synth.c -lm
gcc $SAN -Iinclude -o oracle/libhimut_oracle.so oracle/himut_oracle.c -lm
LD_PRELOAD="$(gcc -print-file-name=libasan.so):$(gcc -print-file-name=libubsan.so)" ASAN_OPTIONS=detect_leaks=0 UBSAN_OPTIONS=print_stacktrace=1 \
  python -m pytest tests/test_bamdec.py tests/test_inflate.py tests/test_thresholds.py tests/test_host.py tests/test_worker_host.py \
  tests/test_oracle_golden.py tests/test_oracle_random.py tests/test_kat.py tests/test_edges.py tests/test_reflib.py \
  tests/test_deflate_conformance.py tests/test_bam_writers.py tests/test_ref_ops.py tests/test_csi.py -q -s -m "not gpu" > /tmp/sanitize_host.log 2>&1 || true
tail -2 /tmp/sanitize_host.log
echo "sanitizer reports: $(grep -c 'runtime error\|AddressSanitizer' /tmp/sanitize_host.log || true)"
grep -A6 'runtime error\|AddressSanitizer' /tmp/sanitize_host.log || true
python -c "import __graft_entry__ as g; g.build(force=True)"
