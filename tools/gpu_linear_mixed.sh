#!/bin/bash
# The 16-bit Linear kernels (DESIGN.md 11.4), in stages that each fit one bounded GPU session:
#   tests     the new GPU tests
#   sites     tools/bench_mixed.py part m (the encoder's Linear sites at 344 064 and 172 032 rows)
#   decoder   tools/bench_mixed.py parts b, c (decoder forward and training step, the linear="autocast" arms with the
#             16-bit Linear kernels on and off)
#   launches  the launch list of the autocast decoder forward (tools/prof_autocast_decoder.py)
# Usage: tools/gpu_linear_mixed.sh [stage ...] (default: all four).  Every stage records the card's name, power limit
# and max SM clock next to its results, in $BENCH_OUT/linear_mixed (default: bench_out/, git-ignored).
OUT="${BENCH_OUT:-bench_out}/linear_mixed"
mkdir -p "$OUT"
STAGES="${*:-tests sites decoder launches}"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee -a "$OUT/card.txt"
for stage in $STAGES; do
  case "$stage" in
    tests)
      timeout 1500 python -m pytest -q -s tests/test_linear_mixed_gpu.py > "$OUT/tests.log" 2>&1
      echo "tests exit $?"
      grep -E "FAILED|Error|passed|failed|grad_w nrel" "$OUT/tests.log" | tail -40 ;;
    sites)
      timeout 1500 python tools/bench_mixed.py --parts m --out "$OUT" > "$OUT/bench_m.log" 2>&1
      echo "sites exit $?"
      grep '"part": "m"' "$OUT/mixed.jsonl" | cut -c1-400 ;;
    decoder)
      timeout 1500 python tools/bench_mixed.py --parts b,c --out "$OUT" > "$OUT/bench_bc.log" 2>&1
      echo "decoder exit $?"
      grep -E '"part": "(b|c)"' "$OUT/mixed.jsonl" | cut -c1-400 ;;
    launches)
      timeout 900 python tools/prof_autocast_decoder.py --out "$OUT" > "$OUT/prof.log" 2>&1
      echo "launches exit $?"
      head -40 "$OUT/decoder_launches.md" ;;
    *) echo "unknown stage $stage"; exit 2 ;;
  esac
done
