#!/bin/bash
# One GPU visit: tests, smoke, bench (all workloads), launch list, full ncu captures of the hot kernels.
set -x
mkdir -p gpurun_out
timeout -k 10 900 python -m pytest tests -m gpu -q --maxfail=60 > gpurun_out/test_full.log 2>&1; tail -3 gpurun_out/test_full.log
timeout -k 10 300 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; tail -2 gpurun_out/smoke.log
timeout -k 10 600 python bench.py --steps 5 --warmup 3 > gpurun_out/bench_c3.json 2> gpurun_out/bench_c3.err; tail -c 600 gpurun_out/bench_c3.json
timeout -k 10 600 python bench.py --steps 3 --warmup 3 --precision bf16 --no-cpu-baseline > gpurun_out/bench_c3_bf16.json 2> gpurun_out/bench_c3_bf16.err
for w in c1 c2 c4; do timeout -k 10 600 python bench.py --workload $w --steps 5 --warmup 3 > gpurun_out/bench_$w.json 2> gpurun_out/bench_$w.err; done
timeout -k 10 600 python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/bench_reference.json 2> gpurun_out/bench_reference.err; tail -c 400 gpurun_out/bench_reference.json
timeout -k 10 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 80 --csv --log-file gpurun_out/launches.csv python tools/profile_step.py bf16x3 6 > gpurun_out/ncu_launch.log 2>&1
timeout -k 10 900 ncu --set full --clock-control none --import-source on -k regex:k_particle_chain_tc -s 2 -c 1 -f -o gpurun_out/prof_chain_tc python tools/profile_step.py bf16x3 4 > gpurun_out/ncu_tc.log 2>&1; tail -1 gpurun_out/ncu_tc.log
timeout -k 10 600 ncu --set full --clock-control none --import-source on -k regex:k_normalize_resample -s 2 -c 1 -f -o gpurun_out/prof_resample python tools/profile_step.py bf16x3 4 > gpurun_out/ncu_nr.log 2>&1; tail -1 gpurun_out/ncu_nr.log
ls -la gpurun_out | head -40
