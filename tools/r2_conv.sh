#!/bin/bash
# round-2 conv kernel check: kernel parity tests, isolated flavour timings
mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_kernels.py -m gpu -x -q -k "conv" 2>&1 | tail -15 > gpurun_out/r2_conv_tests.log
echo "pytest exit=${PIPESTATUS[0]}" >> gpurun_out/r2_conv_tests.log
timeout 300 python tools/bench_conv_flavours.py > gpurun_out/r2_conv_flavours.log 2>&1
echo "exit=$?" >> gpurun_out/r2_conv_flavours.log
