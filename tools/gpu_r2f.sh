#!/bin/bash
# r02: activation-scale tests + engine tests with the new xcorr kernel
mkdir -p gpurun_out
( timeout 900 python -m pytest tests/test_gpu_range.py tests/test_batch_tracker.py -m gpu -q -p no:cacheprovider 2>&1 | tail -60 ) > gpurun_out/r2f_range.log 2>&1
tail -8 gpurun_out/r2f_range.log
( timeout 1500 python -m pytest tests/test_gpu_engine.py tests/test_gpu_shapes.py -m gpu -q -x -p no:cacheprovider 2>&1 | tail -30 ) > gpurun_out/r2f_engine.log 2>&1
tail -4 gpurun_out/r2f_engine.log
