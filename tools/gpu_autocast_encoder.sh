#!/bin/bash
# The autocast encoder: the new GPU tests, tools/bench_mixed.py parts l, p, b, c (the residual + LayerNorm site, the
# 16-bit packed / table forward, the decoder forward and training step with the linear="autocast" arms), then the
# launch list of the autocast decoder forward.  Results go to $BENCH_OUT/autocast (default: bench_out/, git-ignored).
OUT="${BENCH_OUT:-bench_out}/autocast"
mkdir -p "$OUT"
rm -f "$OUT/mixed.jsonl"
timeout 1500 python -m pytest -q tests/test_autocast_encoder_gpu.py tests/test_autocast_linear.py > "$OUT/tests.log" 2>&1
echo "tests exit $?"
grep -E "FAILED|Error|passed|failed" "$OUT/tests.log" | tail -30
timeout 1500 python tools/bench_mixed.py --parts l,p,b,c --out "$OUT" > "$OUT/bench.log" 2>&1
echo "bench exit $?"
tail -3 "$OUT/bench.log"
cut -c1-300 "$OUT/mixed.jsonl"
timeout 900 python tools/prof_autocast_decoder.py --out "$OUT" > "$OUT/prof.log" 2>&1
echo "profile exit $?"
head -30 "$OUT/decoder_launches.md"
