#!/bin/bash
# compute-sanitizer memcheck over a representative subset of the GPU tests (the whole suite under the tool would take too long)
mkdir -p gpurun_out
O=gpurun_out
timeout 1500 compute-sanitizer --tool memcheck --print-limit 10 python -m pytest tests/test_gpu_init.py tests/test_gpu_ba.py tests/test_gpu_coarse.py tests/test_gpu_trace.py tests/test_gpu_marg.py tests/test_gpu_select.py -m gpu -q -x -k "few_points or nf3 or nf4 or small or parity or errors or bit_exact or marg" > $O/san_memcheck.log 2>&1; echo "rc=$?" >> $O/san_memcheck.log
grep -n "passed\|failed\|ERROR SUMMARY\|Invalid\|rc=" $O/san_memcheck.log | cut -c1-200 | tail -12
