#!/bin/bash
# on the GPU box: the evidence set for profiles/ (tests, bench line, reference arm, phase cycles)
python -m pytest tests -m gpu -q 2>&1 | tail -3 > gpurun_out/final_tests.log
python bench.py > gpurun_out/final_bench.json 2> gpurun_out/final_bench.err
python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/final_bench_ref.json 2>> gpurun_out/final_bench.err
python tools/phase_profile.py 64 > gpurun_out/final_phase.txt 2>&1
cat gpurun_out/final_tests.log; head -c 600 gpurun_out/final_bench.json; echo; head -c 400 gpurun_out/final_bench_ref.json
