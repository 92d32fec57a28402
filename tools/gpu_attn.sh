#!/bin/bash
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
timeout 600 python -m pytest tests/test_gpu_kernels.py -q -m gpu -x --timeout 120 -k "attention" 2>&1 | tail -2
timeout 600 python -m pytest tests/test_gpu_decode.py -q -m gpu -x --timeout 300 2>&1 | tail -2
timeout 200 python tools/graph_ab.py 2>&1 | tail -1
timeout 300 python tools/profile_decode.py 4 128 gpurun_out/profile_c2.tsv | tail -1; grep "attention" gpurun_out/profile_c2.tsv | cut -c1-100
timeout 600 python tools/big_decode.py 512 2>&1 | tail -1; grep -E "attention" gpurun_out/profile_big_512.tsv | cut -c1-100
