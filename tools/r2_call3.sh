#!/bin/bash
# round 2, GPU call 3: fixed GLOBAL mode, SELL-U v2 (dedup + batched gathers), lean storage + 512^3 on one GPU, full bench
set -x
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -q -rfEs 2>&1 | tail -40
timeout 300 python tools/cycle_probe.py --n 256 --cycles 36 --time-ops
timeout 600 python tools/async_time.py --n 256 --corrections 35 --reps 2 --variants default,global
( time timeout 1500 python bench.py --impl reference --steps 2 --warmup 1 ) > gpurun_out/bench_r2_call3_ref.json 2> gpurun_out/bench_r2_call3_ref.err; tail -c 1500 gpurun_out/bench_r2_call3_ref.json; tail -4 gpurun_out/bench_r2_call3_ref.err
( time timeout 1500 python bench.py ) > gpurun_out/bench_r2_call3.json 2> gpurun_out/bench_r2_call3.err; tail -c 3000 gpurun_out/bench_r2_call3.json; tail -12 gpurun_out/bench_r2_call3.err
timeout 600 ncu --set full --import-source on --clock-control none -k regex:k_async_amg -c 3 -f -o gpurun_out/prof_r2_async3 \
   python tools/async_time.py --n 256 --corrections 4 --reps 0 --variants default > gpurun_out/prof_r2_async3.log 2>&1 || true
timeout 600 ncu --set full --import-source on --clock-control none -k regex:k_spmv -c 12 -f -o gpurun_out/prof_r2_cycle3 \
   python tools/cycle_probe.py --n 256 --cycles 1 > gpurun_out/prof_r2_cycle3.log 2>&1 || true
ls -la gpurun_out
