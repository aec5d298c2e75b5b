#!/bin/bash
# compute-sanitizer over smoke(), which runs the default tiles for its small batch (single-CTA; the CTA-pair tile
# needs a batch that fills the machine)
mkdir -p gpurun_out
timeout 500 compute-sanitizer --tool memcheck python __graft_entry__.py smoke > gpurun_out/sanitizer_memcheck_pair.log 2>&1
tail -3 gpurun_out/sanitizer_memcheck_pair.log
timeout 500 compute-sanitizer --tool racecheck python __graft_entry__.py smoke > gpurun_out/sanitizer_racecheck_pair.log 2>&1
tail -3 gpurun_out/sanitizer_racecheck_pair.log
