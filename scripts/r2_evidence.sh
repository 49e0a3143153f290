#!/bin/bash
# round-2 evidence pass: parity statistics, scripted success rates, block-size A/B
timeout 600 python tests/parity_report.py > gpurun_out/r2_parity.json 2> gpurun_out/r2_parity.err
timeout 900 python -m pytest tests/test_gpu_scripted.py tests/test_gpu_parity_large.py tests/test_gpu_parity.py -m gpu -q -s 2>&1 | grep -E "scripted|passed|failed|agreement|BASELINE|worst" > gpurun_out/r2_scripted.txt
for v in b64 b32; do echo == $v; PANDA_B200_LIB=$PWD/build_ab/libpanda_$v.so scripts/ab_trees.sh t8$v .; done
