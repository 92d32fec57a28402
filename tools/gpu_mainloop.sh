#!/bin/bash
# main-loop probe: TMA loads and / or MMAs switched off, one HDRVAE_GEMM_DBG setting per process
cd "$(dirname "$0")/.."
for dbg in 0 1 2 3; do HDRVAE_GEMM_DBG=$dbg timeout 300 python tools/mainloop_probe.py; done
