#!/bin/bash
# GPU-box pass: standalone GEMM checks, parity tests, bench.
mkdir -p gpurun_out
timeout 240 python scripts/planes_check.py --bench > gpurun_out/gemm_cluster.txt 2>&1; rc=$?
cat gpurun_out/gemm_cluster.txt >> gpurun_out/gemm_check.txt; echo "rc=$rc" >> gpurun_out/gemm_check.txt
echo "== wide_check" >> gpurun_out/gemm_check.txt
timeout 240 python scripts/wide_check.py --big >> gpurun_out/gemm_check.txt 2>&1; echo "rc=$?" >> gpurun_out/gemm_check.txt
cat gpurun_out/gemm_check.txt
timeout 600 python -m pytest tests -m gpu -x -q > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?" >> gpurun_out/pytest_gpu.log
tail -5 gpurun_out/pytest_gpu.log
timeout 400 python bench.py --steps 10 --warmup 3 > gpurun_out/bench.json 2> gpurun_out/bench.err; cat gpurun_out/bench.json; tail -3 gpurun_out/bench.err
