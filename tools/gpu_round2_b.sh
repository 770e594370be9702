#!/bin/bash
# round-2 GPU pass B: the two tests pass A left red, small-batch (cfg1/2/4 size), cfg5 microbench,
# NIPS bench on the bf16x3 kernels, the ncu launch list of the default bench command
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_fullsize.py tests/test_gpu_update.py -m gpu -q -rA -s -p no:cacheprovider > gpurun_out/pytest_gpu_b.log 2>&1; echo "pytest rc=$?"
grep -E "^parity full-size gradient|^(FAILED|ERROR)|passed|failed" gpurun_out/pytest_gpu_b.log | tail -40
timeout 600 python tools/small_batch.py --out gpurun_out/r02_small_batch.json > gpurun_out/small_batch.log 2>&1; echo "small_batch rc=$?"; tail -5 gpurun_out/small_batch.log
timeout 300 python tools/microbench_cfg5.py > gpurun_out/r02_micro_cfg5.json 2> gpurun_out/micro_cfg5.err; echo "micro rc=$?"; tail -3 gpurun_out/micro_cfg5.err
timeout 600 python bench.py --arch NIPS --steps 20 > gpurun_out/r02_bench_nips_bf16x3_n1.json 2> gpurun_out/bench_nips.err; echo "bench nips rc=$?"; tail -3 gpurun_out/bench_nips.err
python tools/show_bench.py gpurun_out/r02_bench_nips_bf16x3_n1.json 2>&1 | tail -20
timeout 300 python bench.py --steps 2 --warmup 3 --no_cpu_baseline --no_e2e --no_variants > gpurun_out/plain_ncu.log 2>&1 && \
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file gpurun_out/r02_launches_a.csv python bench.py --steps 2 --warmup 3 --no_cpu_baseline --no_e2e --no_variants > gpurun_out/ncu_launch.log 2>&1; echo "ncu launches rc=$?"
