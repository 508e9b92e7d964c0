#!/usr/bin/env bash
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
timeout 900 python -m pytest tests/test_round2_gpu.py tests/test_modules_gpu.py tests/test_fullsize_gpu.py -q -p no:cacheprovider > gpurun_out/r2o_pytest.log 2>&1
grep -n "FAILED\|passed\|failed\|^E  " gpurun_out/r2o_pytest.log | head -20
timeout 300 python bench.py --steps 20 --warmup 5 --no-epoch --no-cpu-baseline --no-aux --no-prop > gpurun_out/r2o_bench_baby.json 2> gpurun_out/r2o_bench_baby.err
python - <<'P'
import json
d=json.loads(open('gpurun_out/r2o_bench_baby.json').read().strip().splitlines()[-1])
print('value=%.4g ms=%.3f e2e=%.4g'%(d['value'],d['ms_per_step'],d['e2e']['value']))
print('variants', json.dumps(d.get('variants'))[:600])
print('roofline', round(d['roofline']['frac'],3), {k:(round(v['avg_ms'],4),round(v['tflops'])) for k,v in d['roofline']['by_shape_MxNxK'].items()})
print('breakdown',{k:v['ms_per_step'] for k,v in d['breakdown_ms_per_step'].items()})
P
python tools/bench_spmm.py baby | tail -2
python tools/bench_spmm.py sports | tail -2
