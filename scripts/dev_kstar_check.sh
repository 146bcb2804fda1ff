#!/bin/bash
# after a K* arithmetic change: the parity tests that exercise K* (all four kernel families, training points as
# candidates, goldens, full-size spot checks), then the bench without its side measurements
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_parity.py tests/test_golden.py tests/test_gpu_fullsize.py tests/test_gpu_split.py tests/test_kg.py tests/test_gpu_kernel_list.py -m gpu -x -q > gpurun_out/kstar_tests.log 2>&1
echo "tests rc=$?"; tail -3 gpurun_out/kstar_tests.log
timeout 300 python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-mixed --no-extras > gpurun_out/bench_kstar.json 2> gpurun_out/bench_kstar.err
echo "bench rc=$?"
python -c "
import json; d=json.load(open('gpurun_out/bench_kstar.json')); print(round(d['value']), round(d['ms_per_step'],1), {k:round(v/3,1) for k,v in d['roofline']['kernel_ms'].items()}, d['clocks']['sm_mhz'])"
