#!/usr/bin/env bash
# round-2 job A: full GPU test suite + bench lines of the new top-k / q_sample paths
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
nvidia-smi --query-gpu=name,clocks.max.sm,power.limit --format=csv > gpurun_out/r2a_gpu.txt 2>&1
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider > gpurun_out/r2a_pytest.log 2>&1
echo "pytest rc=$?" >> gpurun_out/r2a_pytest.log
timeout 600 python bench.py --steps 10 --warmup 3 > gpurun_out/r2a_bench_baby.json 2> gpurun_out/r2a_bench_baby.err
echo "bench rc=$?"
timeout 300 python bench.py --steps 10 --warmup 3 --sampling-step 0 --no-epoch --no-cpu-baseline --no-aux > gpurun_out/r2a_bench_baby_ss0.json 2> gpurun_out/r2a_bench_baby_ss0.err
timeout 300 python bench.py --steps 10 --warmup 3 --workload sports --no-epoch --no-cpu-baseline --no-aux > gpurun_out/r2a_bench_sports.json 2> gpurun_out/r2a_bench_sports.err
timeout 400 python bench.py --steps 4 --warmup 3 --workload scaleout --no-epoch --no-cpu-baseline --no-aux > gpurun_out/r2a_bench_scaleout.json 2> gpurun_out/r2a_bench_scaleout.err
tail -5 gpurun_out/r2a_pytest.log
