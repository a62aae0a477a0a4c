#!/bin/bash
# Builds the GPU probe binaries in-tree (git-ignored).
set -e
cd "$(dirname "$0")"
F="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17"
nvcc $F conv_probe.cu ../lungmask_b200/csrc/conv_tc.cu -o conv_probe -lcuda
nvcc $F -DLM_CONV_PROFILE conv_probe.cu ../lungmask_b200/csrc/conv_tc.cu -o conv_probe_prof -lcuda
[ -f umma_probe.cu ] && nvcc $F umma_probe.cu -o umma_probe -lcuda || true
ls -la conv_probe conv_probe_prof
