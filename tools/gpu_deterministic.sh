#!/bin/bash
# Deterministic mode: the new GPU tests, then tools/bench_deterministic.py (flag off against flag on).
# Results go to $BENCH_OUT/deterministic (default: bench_out/, git-ignored).
OUT="${BENCH_OUT:-bench_out}/deterministic"
mkdir -p "$OUT"
rm -f "$OUT/deterministic.jsonl"
timeout 1200 python -m pytest -q -s tests/test_deterministic_gpu.py > "$OUT/tests.log" 2>&1
echo "tests exit $?"
tail -5 "$OUT/tests.log"
timeout 1200 python tools/bench_deterministic.py --out "$OUT" > "$OUT/bench.log" 2>&1
echo "bench exit $?"
cut -c1-600 "$OUT/deterministic.jsonl"
