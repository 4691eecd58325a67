#!/bin/bash
set -u
mkdir -p gpurun_out
make -C kubebrain_b200/csrc 2>&1 | tail -2
echo "== quick tests"; timeout -s KILL 900 python -m pytest tests/test_gpu_round2.py tests/test_cpp_host.py -x -q -m gpu -k "not geometries" 2>&1 | tail -6 | tee gpurun_out/t_r2.log
timeout -s KILL 600 python -m pytest tests/test_gpu_parity.py -x -q -k "fanout or config3 or watch or compact or config4_shape or fuzz_range or config2_shape or range_table" 2>&1 | tail -8 | tee gpurun_out/t_fanout.log
echo "== bench"; timeout -s KILL 1200 python bench.py --steps 20 --warmup 5 > gpurun_out/bench.json 2> gpurun_out/bench.err; echo "rc=$?"; tail -c 1500 gpurun_out/bench.err
python - <<'PY'
import json
try:
    d=json.loads([l for l in open('gpurun_out/bench.json') if l.startswith('{')][-1])
    print({k:d[k] for k in ('value','ms_per_step','parity_checked','gpu_launches')}, d['e2e'])
    print('latency', d.get('latency')); print('fanout_alone', d.get('fanout_alone'))
    print('compaction', {k:v for k,v in d['extra']['compaction'].items()})
    for k in d['kernels'][:12]: print(k['name'], round(k['avg_us'],1), round(k['achieved_gbs'] or 0,1), round(k['share'],3))
    print(d['host_call_us']); print([(k['name'],round(k['avg_us'])) for k in d['host_segments']])
except Exception as e: print('bench parse failed', e)
PY
echo "== all gpu tests"; timeout -s KILL 1500 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 | tee gpurun_out/t_gpu.log
