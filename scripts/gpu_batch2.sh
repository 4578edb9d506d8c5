mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_made_inverse.py -m gpu -q --timeout 300 > gpurun_out/made_inv_tests.log 2>&1; echo "inverse pytest rc=$?"; grep -E "passed|failed|^FAILED" gpurun_out/made_inv_tests.log | tail -5
timeout 300 python scripts/bench_made_inverse.py 4096 32768 262144 > gpurun_out/made_inv_bench.log 2>&1; echo "bench rc=$?"; cut -c1-330 gpurun_out/made_inv_bench.log | tail -4
timeout 600 python -m pytest tests/test_gpu_parity.py -m gpu -q --timeout 300 -k "actnorm" 2>&1 | tail -3
