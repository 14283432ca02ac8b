#!/bin/bash
# round 2, run B (2+ GPUs): train tests, phase stamps, DP tests, DP stamps (multicast on/off), bench N=1,2
N=${1:-2}
mkdir -p gpurun_out; rm -f gpurun_out/summary.txt
S=gpurun_out/summary.txt
timeout 900 python -m pytest tests/test_gpu_train.py tests/test_gpu_forward.py -q -m gpu --tb=short -x > gpurun_out/pytest_train.log 2>&1; echo "train tests exit $?" >> $S
tail -5 gpurun_out/pytest_train.log >> $S
timeout 200 python tools/phase_timing.py > gpurun_out/phase_n1.log 2>&1; echo "phase n1 exit $?" >> $S; grep -E "steady state \(graph replay, rep 2\)|us/step|   setup" gpurun_out/phase_n1.log | tail -4 >> $S
timeout 600 python -m pytest tests/test_gpu_dp.py -q -m gpu --tb=short -x > gpurun_out/test_gpu_dp.log 2>&1; echo "dp tests exit $?" >> $S
tail -8 gpurun_out/test_gpu_dp.log >> $S
for MC in 1 0; do
  B2H_MULTICAST=$MC timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29541 tools/phase_timing.py > gpurun_out/phase_n${N}_mc$MC.log 2>&1; echo "phase n$N mc$MC exit $?" >> $S
  grep -E "exchange=|rep 2|us/step|   setup" gpurun_out/phase_n${N}_mc$MC.log | tail -12 >> $S
done
timeout 300 python bench.py --steps 20 --warmup 5 --skip-extras > gpurun_out/bench_n1.json 2> gpurun_out/bench_n1.err; echo "bench n1 exit $?" >> $S
timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533 bench.py --gpus $N --steps 20 --warmup 5 > gpurun_out/bench_n$N.json 2> gpurun_out/bench_n$N.err; echo "bench n$N exit $?" >> $S
tail -3 gpurun_out/bench_n$N.err >> $S
timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29534 bench.py --gpus $N --steps 20 --warmup 5 --no-multicast > gpurun_out/bench_n${N}_nomc.json 2> gpurun_out/bench_n${N}_nomc.err; echo "bench n$N nomc exit $?" >> $S
python - <<PY >> $S 2>&1
import json
for f in ('bench_n1', 'bench_n$N', 'bench_n${N}_nomc'):
    try:
        d = json.load(open('gpurun_out/%s.json' % f))
        print(f, d['n_gpus'], 'value', d['value'], 'us/step', d['ms_per_step'] * 1e3, 'e2e', d['e2e']['value'], 'e2e us', d['e2e']['us_per_step'], d.get('dp_parity'), d.get('tc_status'), d.get('status_ok'))
    except Exception as e:
        print(f, 'ERR', e)
PY
cat $S
