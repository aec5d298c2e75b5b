#!/bin/bash
# r02: convergent-issue GEMM kernels — op tests, shape tests, whole GPU suite, tracker tests, bench with launch list
mkdir -p gpurun_out
( timeout 900 python -m pytest tests/test_gpu_ops.py -m gpu -q -x -p no:cacheprovider 2>&1 | tail -15 ) > gpurun_out/r2d_ops.log 2>&1
tail -3 gpurun_out/r2d_ops.log
( timeout 900 python -m pytest tests/test_gpu_shapes.py tests/test_batch_tracker.py -m gpu -q -p no:cacheprovider 2>&1 | tail -40 ) > gpurun_out/r2d_shapes.log 2>&1
tail -5 gpurun_out/r2d_shapes.log
( timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider --deselect tests/test_gpu_shapes.py --deselect tests/test_gpu_ops.py --deselect tests/test_batch_tracker.py 2>&1 | tail -30 ) > gpurun_out/r2d_pytest.log 2>&1
tail -3 gpurun_out/r2d_pytest.log
timeout 1200 python bench.py --steps 20 --warmup 3 --dump-layers gpurun_out/r2d_layers.tsv > gpurun_out/r2d_bench.json 2> gpurun_out/r2d_bench.err
tail -3 gpurun_out/r2d_bench.err; cut -c1-300 gpurun_out/r2d_bench.json
