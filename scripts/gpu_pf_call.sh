#!/bin/bash
# hoisted-load / branch-free-reciprocal variants of RevA, RevC (ONE B200): default (6 CTAs/SM, 80 regs), 5 and 4 CTAs/SM builds
tag=${1:-r02e}
mkdir -p gpurun_out
export KB_QUIET=1 KB_NJ=720 KB_TILE=16x12
timeout 200 python -m pytest tests/test_gpu_parity.py -m gpu -q -x -p no:cacheprovider 2>&1 | tail -2
timeout 300 python scripts/kbench.py dafoam_b200/libdab200.so dafoam_b200/libdab200_mb5.so dafoam_b200/libdab200_mb4.so 2>&1 | tail -3
ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k 'regex:Rev[ABC]' -s 6 -c 3 -f -o gpurun_out/${tag}_rev \
    python scripts/kbench.py > gpurun_out/${tag}_rev.log 2>&1
ncu -i gpurun_out/${tag}_rev.ncu-rep --page raw --csv > gpurun_out/${tag}_rev_raw.csv 2>/dev/null
ls -la gpurun_out | tail -3
