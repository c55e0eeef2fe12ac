#!/bin/bash
O=gpurun_out; mkdir -p $O
timeout 900 python -m pytest tests/test_gpu_ba.py -x -q -m gpu > $O/r02_pytest6.log 2>&1; echo "pytest rc=$?" >> $O/r02_pytest6.log
COVINS_SKIP_CPU_BASELINE=1 timeout 600 python bench.py --steps 10 --warmup 3 > $O/r02_bench3.json 2> $O/r02_bench3.err
COVINS_B200_NO_CHAIN_STREAM=1 COVINS_SKIP_CPU_BASELINE=1 timeout 600 python bench.py --steps 10 --warmup 3 > $O/r02_bench3_nochain.json 2> $O/r02_bench3_nochain.err
tail -3 $O/r02_pytest6.log; python - <<'PY'
import json
for f in ("r02_bench3.json", "r02_bench3_nochain.json"):
    try:
        d = json.loads(open("gpurun_out/" + f).read().strip().splitlines()[-1])
        print(f, d["value"], d["phase_ms_per_step"], d["match"]["value"], d["match"]["roofline"]["frac"], d["match"]["e2e"]["value"], d["pgo"]["value"], d["match"]["sift_l2"]["value"])
    except Exception as e:
        print(f, "ERR", e)
PY
tail -3 $O/r02_bench3.err
