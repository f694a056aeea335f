#!/bin/bash
# usage (on the GPU box): bash tools/gpu_round.sh <tag> [ncu]   -> GPU tests, default bench (device-resident only), optional ncu capture of K2
T=$1
python -m pytest tests -m gpu -x -q > gpurun_out/gputests_$T.log 2>&1; tail -2 gpurun_out/gputests_$T.log
summ() { python -c "
import json,sys;d=json.load(open(sys.argv[1]));print(sys.argv[1], round(d['value']),{k:round(v['avg_ms'],4) for k,v in d['kernels'].items()})" $1; }
python bench.py --no-e2e --no-cpu-baseline --no-overlap --no-extras --no-other-configs --sustain-seconds 0 --parity-frames 0 > gpurun_out/bench_$T.json 2> gpurun_out/bench_$T.err; summ gpurun_out/bench_$T.json
if [ "$2" = ncu ]; then
ncu --set full --clock-control none --import-source on -k regex:fdct_quant -s 1 -c 1 -o gpurun_out/prof_$T -f python bench.py --no-e2e --no-cpu-baseline --no-overlap --no-extras --no-other-configs --sustain-seconds 0 --parity-frames 0 --frames 64 --steps 1 --warmup 1 > gpurun_out/ncu_$T.log 2>&1
fi
