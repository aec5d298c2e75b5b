#!/bin/bash
mkdir -p gpurun_out
timeout 600 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k regex:xcorr_nhwc -s 4 -c 1 -f -o gpurun_out/prof_xcorr_nhwc_r02 python bench.py --steps 1 --warmup 3 --min-seconds 0 --no-cpu --no-context --no-verify --no-loop > gpurun_out/r2h_ncu_xcorr.log 2>&1
tail -2 gpurun_out/r2h_ncu_xcorr.log | cut -c1-200
