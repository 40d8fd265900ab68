#!/bin/bash
# Ablation build (-DTIC_ABLATE: TIC_DBG stage switches, wait-time counters) next to the shipped library:
# tf_image_compression_b200/libtic_ablate.so.  tools/fused_ablate.py and tools/fused_waits.py load it; the package never does.
cd "$(dirname "$0")/.." && nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -shared -Xcompiler -fPIC -DTIC_ABLATE -o tf_image_compression_b200/libtic_ablate.so tf_image_compression_b200/csrc/tic_api.cu -lcuda > /tmp/ablate_build.log 2>&1
rc=$?; grep -E "rror" /tmp/ablate_build.log | head; echo "ablate build rc=$rc"; exit $rc
