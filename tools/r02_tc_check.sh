#!/bin/bash
O=gpurun_out; mkdir -p $O
timeout 240 python -m pytest tests/test_gpu_matching.py tests/test_gpu_tc_match.py tests/test_shim.py -x -q -m gpu --timeout 60 > $O/r02_pytest5.log 2>&1; echo "pytest rc=$?" >> $O/r02_pytest5.log
tail -3 $O/r02_pytest5.log
