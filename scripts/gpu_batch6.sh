python scripts/bench_made_inverse.py 4096 32768 2>/dev/null | cut -c1-260
timeout 600 python -m pytest tests/test_gpu_parity.py -m gpu -q --timeout 300 -k "actnorm" 2>&1 | tail -2
python scripts/bench_kernels.py 2>/dev/null | grep actnorm | cut -c1-200
