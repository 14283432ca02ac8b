#!/bin/bash
# N=1: K0 (preprocessing) parity + graph-replay timings per clip length + bench sections
mkdir -p gpurun_out; rm -f gpurun_out/summary.txt
S=gpurun_out/summary.txt
timeout 900 python -m pytest tests/test_gpu_preprocess.py tests/test_gpu_forward.py -q -m gpu --tb=short > gpurun_out/pytest_k0.log 2>&1; echo "k0+fwd tests exit $?" >> $S
tail -3 gpurun_out/pytest_k0.log >> $S
python tools/k0_prof.py time 27000 108000 216000 864000 2>&1 | grep "us/launch" >> $S
timeout 300 python bench.py --steps 20 --warmup 5 > gpurun_out/bench_k0.json 2> gpurun_out/bench_k0.err; echo "bench exit $?" >> $S
python - <<PY >> $S 2>&1
import json
d = json.load(open('gpurun_out/bench_k0.json'))
print('train us/step', d['ms_per_step'] * 1e3, 'fwd', d['fwd'].get('ms_per_batch'))
print('preprocess', d['preprocess']['ms_per_launch'], d['preprocess']['roofline']['frac'])
print('stream16', d['stream']['stride16'].get('unique_frames_per_sec'), 'stream64', d['stream']['stride64'].get('unique_frames_per_sec'))
PY
cat $S
