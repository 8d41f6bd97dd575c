#!/bin/bash
# Round-2 evidence visit (one B200): parity suite, bench (both arms), ncu launch list, ncu --set full of the three new / changed
# kernel families, size sweep.
# usage (under gpurun): bash tools/gpu_round2.sh TAG
TAG=${1:-r2}; OUT=gpurun_out; mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $OUT/smi_$TAG.txt; nproc > $OUT/nproc_$TAG.txt
timeout -s KILL 600 python -m pytest tests -m gpu -q --durations=5 > $OUT/pytest_gpu_$TAG.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_gpu_$TAG.log
timeout -s KILL 600 python bench.py --steps 20 --warmup 3 > $OUT/bench_$TAG.json 2> $OUT/bench_$TAG.err; echo "bench rc=$?" >> $OUT/bench_$TAG.err
timeout -s KILL 600 python bench.py --impl reference --steps 3 --warmup 1 > $OUT/bench_ref_$TAG.json 2>> $OUT/bench_$TAG.err
timeout -s KILL 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches_$TAG.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu --no-configs > $OUT/ncu_launch_$TAG.log 2>&1
timeout -s KILL 400 ncu --set full --clock-control none --import-source on -k regex:render_r64 -s 3 -c 1 -f -o $OUT/prof_r64_$TAG \
    python bench.py --steps 2 --warmup 3 --no-cpu --no-configs > $OUT/ncu_full_r64_$TAG.log 2>&1
timeout -s KILL 400 ncu --set full --clock-control none --import-source on -k regex:render_w_ -s 3 -c 1 -f -o $OUT/prof_w_$TAG \
    python tools/sweep.py X:CS16:512:1:26 1 > $OUT/ncu_full_w_$TAG.log 2>&1
SP_FOURSTEP=ring timeout -s KILL 400 ncu --set full --clock-control none --import-source on -k regex:render_big -s 3 -c 1 -f -o $OUT/prof_big_$TAG \
    python tools/sweep.py C5 1 > $OUT/ncu_full_big_$TAG.log 2>&1
CASES=$(for n in 64 128 256 512 1024 2048 4096 8192 16384 32768 65536 131072; do echo -n "X:CS16:$n:1:26,"; done)
timeout -s KILL 600 python tools/sweep.py ${CASES}C1,C2,C2-hann,C2-z2,C2-z4,C2-z8 5 > $OUT/sweep_$TAG.jsonl 2> $OUT/sweep_$TAG.err
tail -3 $OUT/pytest_gpu_$TAG.log; cut -c1-400 $OUT/bench_$TAG.json; tail -3 $OUT/bench_$TAG.err; ls -la $OUT | tail -25
