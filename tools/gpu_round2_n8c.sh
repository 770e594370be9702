#!/bin/bash
# round 2, 8 GPUs of one box: where does the N = 8 step lose against N = 1?  The tail all-reduce on a communicator limited to the
# reserved SMs (new default) vs NCCL's default channel count (PAACB_TAIL_MAX_CTAS=0), one all-reduce after the whole backward;
# preceded by N = 1 on the same box and the 8-rank == 1-rank update check on the new default.
mkdir -p gpurun_out
OUT=gpurun_out/r02_n8_tail_allreduce.txt
: > $OUT
run() {  # label, env..., -- extra bench args
  label=$1; shift
  env "$@" timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29563 bench.py --gpus 8 --steps 30 --no_e2e --no_variants $EXTRA > gpurun_out/n8c.json 2> gpurun_out/n8c.err || tail -3 gpurun_out/n8c.err >> $OUT
  python - >> $OUT <<PY
import json
try:
    d=json.loads(open('gpurun_out/n8c.json').read().strip().splitlines()[-1])
    ks={x['name']:x['ms']/d['steps'] for x in d['kernels']}
    print('%-58s ms/step %.3f  value %.2f M  conv3_wgrad %.3f conv2_wgrad %.3f conv1_wgrad %.3f  clocks %s %s' % ('$label', d['ms_per_step'], d['value']/1e6, ks['conv3_wgrad'], ks['conv2_wgrad'], ks['conv1_wgrad'], d['clocks']['sm_mhz'], d['clocks']['reasons']))
except Exception as e:
    print('$label failed', e)
PY
}
timeout 300 python bench.py --steps 30 --no_cpu_baseline --no_variants --no_e2e > gpurun_out/n8c_n1.json 2> gpurun_out/n8c.err
python - >> $OUT <<PY
import json
d=json.loads(open('gpurun_out/n8c_n1.json').read().strip().splitlines()[-1])
ks={x['name']:x['ms']/d['steps'] for x in d['kernels']}
print('%-58s ms/step %.3f  value %.2f M  conv3_wgrad %.3f conv2_wgrad %.3f conv1_wgrad %.3f  clocks %s %s' % ('N = 1, same box', d['ms_per_step'], d['value']/1e6, ks['conv3_wgrad'], ks['conv2_wgrad'], ks['conv1_wgrad'], d['clocks']['sm_mhz'], d['clocks']['reasons']))
PY
PAACB_CHECK_MATH=bf16x3 timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29533 tools/multi_gpu_check.py 2>&1 | grep "multi_gpu_check" >> $OUT
EXTRA=""
run "N = 8, tail on 8 CTAs, 8 SMs reserved (default)" PAACB_X=1
run "N = 8, tail on NCCL's default channels (round-2 behaviour)" PAACB_TAIL_MAX_CTAS=0
EXTRA="--no_overlap_allreduce"
run "N = 8, one all-reduce after the whole backward" PAACB_X=1
cat $OUT
