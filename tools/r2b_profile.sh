#!/bin/bash
# ncu evidence of the int8 pre-filtered chain (after the same command has exited 0 without ncu):
# launch list of two timed steps + --set full of the two scans, 10 M rows, 1 GPU
mkdir -p gpurun_out/r2b
B="python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-stages --parity-queries 0"
$B > gpurun_out/r2b/prof_plain.json 2> gpurun_out/r2b/prof_plain.err; echo "plain rc=$?"
ncu --metrics gpu__time_duration.sum --clock-control none \
    -k regex:"dense_|bm25|merge|fuse|rescore|pack_|finalize" -s 721 -c 28 --csv \
    --log-file gpurun_out/r2b/launches_q8.csv $B > gpurun_out/r2b/ncu_list.log 2>&1; echo "list rc=$?"
ncu --set full --clock-control none --import-source on -k regex:"dense_scan|bm25_scan" -s 200 -c 2 \
    -o gpurun_out/r2b/scan_q8_full -f $B > gpurun_out/r2b/ncu_full.log 2>&1; echo "full rc=$?"
ls -la gpurun_out/r2b/*.ncu-rep
