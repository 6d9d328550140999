#!/bin/bash
# GroupNorm training path: the new GPU tests, then tools/bench_decoder_train.py (kernel level + whole decoder step).
# Results go to $BENCH_OUT/decoder_train (default: bench_out/, git-ignored).
OUT="${BENCH_OUT:-bench_out}/decoder_train"
mkdir -p "$OUT"
rm -f "$OUT/decoder_train.jsonl"
timeout 900 python -m pytest -q -s tests/test_group_norm_train_gpu.py > "$OUT/tests.log" 2>&1
echo "tests exit $?"
tail -3 "$OUT/tests.log"
timeout 1200 python tools/bench_decoder_train.py --out "$OUT" > "$OUT/bench.log" 2>&1
echo "bench exit $?"
cut -c1-400 "$OUT/decoder_train.jsonl"
