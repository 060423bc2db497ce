#!/bin/bash
mkdir -p gpurun_out
timeout 1200 python -m pytest tests -q -m gpu > gpurun_out/r02_gpu_all.log 2>&1; echo "all gpu tests exit $?: $(tail -n 4 gpurun_out/r02_gpu_all.log)"
python tools/prof_tc.py 512 5 2 cont > gpurun_out/r02_cont_prof.log 2>&1; tail -2 gpurun_out/r02_cont_prof.log
