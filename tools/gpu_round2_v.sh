#!/bin/bash
# round 2, pass V: conv3 forward with two samples per tile -- parity, then same-box A/B by environment knob
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_tc.py tests/test_gpu_forward.py -m gpu -q -x -p no:cacheprovider 2>&1 | tail -5; echo "pytest rc=${PIPESTATUS[0]}"
for rep in 1 2; do for K in 0 1; do
PAACB_CONV3_PACKED=$K timeout 300 python bench.py --steps 20 --no_cpu_baseline --no_variants --no_e2e > gpurun_out/c3p_$K.json 2> gpurun_out/c3p.err || tail -5 gpurun_out/c3p.err
python - <<PY
import json
d=json.loads(open('gpurun_out/c3p_$K.json').read().strip().splitlines()[-1])
ks={x['name']:x['ms']/d['steps'] for x in d['kernels']}
print('packed=$K ms/step %.3f'%d['ms_per_step'], ' '.join('%s %.3f'%(k,ks[k]) for k in ('conv3_fwd','conv2_fwd','fc4_fwd')), 'loss %.6f'%d['loss'], 'clocks', d['clocks']['sm_mhz'])
PY
done; done
