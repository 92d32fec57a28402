#!/bin/bash
mkdir -p gpurun_out
( timeout 900 python -m pytest tests -m gpu -q -x ) > gpurun_out/r2i_pytest.log 2>&1
echo "pytest rc=$?"; tail -4 gpurun_out/r2i_pytest.log | cut -c1-600
timeout 300 python tools/attn_bench.py 1x4096 1x16384 4x16384 1x65536 2>&1
