#!/bin/bash
# AddressSanitizer + UBSan over the kernels' tile programs: csrc/hostsim.cpp runs the SAME __host__ __device__ code as the
# CUDA build (swt2_core.cuh: every planned pass form and both uint8 staging forms; hamming_core.cuh: stage A / S / B,
# stash and walk forms, shard scans), thread by thread, with the shared-memory buffers as exactly-sized heap blocks — so an out-of-range shared / global
# index of those programs is an ASan report here.  compute-sanitizer itself is closed on this project's GPU pool
# (profiles/r2_sanitizer.md).  Run in the build container:   bash tools/sim_asan.sh
set -e
cd "$(dirname "$0")/.."
OUT=/tmp/libb200ret_sim_asan.so
g++ -O1 -g -std=c++17 -fPIC -shared -fsanitize=address,undefined -fno-sanitize-recover=undefined -fno-omit-frame-pointer \
    -Wall -Wno-unknown-pragmas -I include -I image_retrieval_wavelet_b200/csrc -o $OUT image_retrieval_wavelet_b200/csrc/hostsim.cpp
ASAN=$(g++ -print-file-name=libasan.so)
B200RET_SIM_LIB=$OUT LD_PRELOAD=$ASAN ASAN_OPTIONS=detect_leaks=0:abort_on_error=0:exitcode=97 \
    python -m pytest tests/test_sim_kernels.py tests/test_dist_gloo.py -x -q -p no:cacheprovider "$@"
