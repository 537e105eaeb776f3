#!/bin/bash
# usage: tools/e2e_stream_sweep.sh > gpurun_out/e2e_stream_sweep.txt
for B in 1024 4096 16384; do timeout 120 python tools/e2e_stream_sweep.py $B; done
