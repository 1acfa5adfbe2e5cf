#!/bin/bash
# Round profile set (run under gpurun): bench line, ncu launch list of the same command, full captures of the
# front-end and CMVN kernels at the bench workload.  $1 = tag
TAG=${1:-r01}
mkdir -p gpurun_out
python bench.py > gpurun_out/bench_$TAG.json 2> gpurun_out/bench_$TAG.err
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches_$TAG.csv \
    python bench.py --steps 2 --warmup 1 > gpurun_out/bench_under_ncu_$TAG.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:frontend_r16 -s 3 -c 1 \
    -o gpurun_out/prof_fe_$TAG -f python scripts/quick_time.py 1024 > gpurun_out/ncu_fe_$TAG.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:cmvn_staged -s 3 -c 1 \
    -o gpurun_out/prof_cmvn_$TAG -f python scripts/quick_time.py 1024 > gpurun_out/ncu_cmvn_$TAG.log 2>&1
cat gpurun_out/bench_$TAG.json
ncu --set full --clock-control none -k "regex:tdnn_tc_(pair|stats)_kernel" -s 14 -c 7 \
    -o gpurun_out/prof_tdnn_$TAG -f python bench.py --workload tdnn --steps 3 --warmup 1 --no-stages --no-cpu-baseline > gpurun_out/ncu_tdnn_$TAG.log 2>&1
python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/bench_ref_$TAG.json 2> gpurun_out/bench_ref_$TAG.err
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke_$TAG.log 2>&1; tail -2 gpurun_out/smoke_$TAG.log
ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file gpurun_out/launches_w2x_$TAG.csv \
    python bench.py --workload wav2xvec --steps 2 --warmup 1 --no-stages --no-cpu-baseline > gpurun_out/bench_w2x_under_ncu_$TAG.log 2>&1
