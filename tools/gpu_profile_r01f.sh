#!/bin/bash
# Round-1 (f) evidence run on the final tree: launch list of the bench command, full captures of k_accumulate (2^20),
# and of the batched look-up sum in config-3 mode (after the instruction-cache fix).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:k_ -c 600 --csv --log-file gpurun_out/launches_bench_f.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline --sweep "" > gpurun_out/bench_under_ncu_f.log 2>&1
SIZES=20 NOPINT=1 timeout 900 ncu --set full --clock-control none --import-source on -k regex:k_accumulate -s 2 -c 1 \
     -f -o gpurun_out/prof_f_k_accumulate_20 python tools/quick_bench.py > gpurun_out/ncu_f_acc.log 2>&1
NB=2048 WINDOWS=0 timeout 900 ncu --set full --clock-control none --import-source on -k regex:k_lut_sum -s 1 -c 1 -f \
     -o gpurun_out/prof_f_k_lut_sum_cfg3 python tools/config34.py > gpurun_out/ncu_f_cfg3.log 2>&1
ls -la gpurun_out/prof_f_*.ncu-rep
