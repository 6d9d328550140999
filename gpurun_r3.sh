timeout 900 python -m pytest -q tests/test_mixed_precision_gpu.py tests/test_parity_gpu.py tests/test_deterministic_gpu.py -p no:cacheprovider 2>&1 | grep -E "^FAILED|passed|failed" | tail -15
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 2>&1 | tail -1 | cut -c1-200
