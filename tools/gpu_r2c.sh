#!/bin/bash
mkdir -p gpurun_out
( timeout 900 python -m pytest tests/test_batch_tracker.py -m gpu -q -x -p no:cacheprovider 2>&1 | tail -30 ) > gpurun_out/r2c_tracker.log 2>&1
tail -5 gpurun_out/r2c_tracker.log
timeout 600 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k regex:conv3x3_patch -s 2 -c 1 -f -o gpurun_out/prof_patch64_r02 python tools/exp_patch.py > gpurun_out/r2c_ncu_patch.log 2>&1
tail -2 gpurun_out/r2c_ncu_patch.log | cut -c1-200
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r2c_patch_launches.csv python tools/exp_patch.py > /dev/null 2>&1
