#!/bin/bash
# Mixed precision: the new GPU tests, then tools/bench_mixed.py (the op in fp32 / bf16 / fp16, the decoder under
# autocast).  Results go to $BENCH_OUT/mixed (default: bench_out/, git-ignored).
OUT="${BENCH_OUT:-bench_out}/mixed"
mkdir -p "$OUT"
rm -f "$OUT/mixed.jsonl"
timeout 1500 python -m pytest -q tests/test_mixed_precision_gpu.py > "$OUT/tests.log" 2>&1
echo "tests exit $?"
grep -E "FAILED|Error|passed|failed" "$OUT/tests.log" | tail -30
timeout 1500 python tools/bench_mixed.py --out "$OUT" > "$OUT/bench.log" 2>&1
echo "bench exit $?"
tail -3 "$OUT/bench.log"
cut -c1-400 "$OUT/mixed.jsonl"
