#!/bin/bash
# Round-2 single-GPU validation: GPU test-suite, bench line; logs go to $O.
O=gpurun_out; mkdir -p $O
timeout 900 python -m pytest tests -x -q -m gpu > $O/r02_pytest4.log 2>&1; echo "pytest rc=$?" >> $O/r02_pytest4.log
COVINS_SKIP_CPU_BASELINE=1 timeout 600 python bench.py --steps 10 --warmup 3 > $O/r02_bench2.json 2> $O/r02_bench2.err
tail -3 $O/r02_pytest4.log; tail -c 600 $O/r02_bench2.json
