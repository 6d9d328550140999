#!/bin/bash
# The 16-bit GroupNorm kernels (DESIGN.md 11.3), in stages that each fit one bounded GPU session:
#   tests     the new GPU tests
#   sites     tools/bench_mixed.py part g (the GroupNorm sites of the decoder at 1024x2048, batch 8)
#   decoder   tools/bench_mixed.py parts b, c (decoder forward and training step, the linear="autocast" arms with the
#             16-bit GroupNorm kernels on and off)
#   launches  the launch list of the autocast decoder forward (tools/prof_autocast_decoder.py)
# Usage: tools/gpu_group_norm_mixed.sh [stage ...] (default: all four).  Every stage records the card's name and power
# limit next to its results, in $BENCH_OUT/gn_mixed (default: bench_out/, git-ignored).
OUT="${BENCH_OUT:-bench_out}/gn_mixed"
mkdir -p "$OUT"
STAGES="${*:-tests sites decoder launches}"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee -a "$OUT/card.txt"
for stage in $STAGES; do
  case "$stage" in
    tests)
      timeout 1500 python -m pytest -q -s tests/test_group_norm_mixed_gpu.py > "$OUT/tests.log" 2>&1
      echo "tests exit $?"
      grep -E "FAILED|Error|passed|failed|decoder, 16-bit" "$OUT/tests.log" | tail -30 ;;
    sites)
      timeout 1500 python tools/bench_mixed.py --parts g --out "$OUT" > "$OUT/bench_g.log" 2>&1
      echo "sites exit $?"
      grep '"part": "g"' "$OUT/mixed.jsonl" | cut -c1-400 ;;
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
