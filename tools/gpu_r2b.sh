#!/bin/bash
# r02: bulk xcorr tests, then the r2a sequence
mkdir -p gpurun_out
( timeout 600 python -m pytest tests/test_gpu_ops.py -m gpu -q -p no:cacheprovider -k "xcorr" 2>&1 | tail -15 ) > gpurun_out/r2b_xcorr.log 2>&1
tail -4 gpurun_out/r2b_xcorr.log
bash tools/gpu_r2a.sh
timeout 300 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k regex:xcorr_bulk -s 4 -c 1 -f -o gpurun_out/prof_xcorr_bulk_r02 python tools/exp_xcorr.py > gpurun_out/r2b_ncu_xcorr.log 2>&1
tail -2 gpurun_out/r2b_ncu_xcorr.log | cut -c1-200
