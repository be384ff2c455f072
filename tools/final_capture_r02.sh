#!/bin/bash
# Round-2 captures (run under gpurun, one GPU): bench line, reference arm, ncu launch list of the bench command, ncu --set full of the
# traversal + shading kernels of one C2 pass run as a single path range, per-stage times, per-warp timelines.
T=${1:-s1}
O=gpurun_out
mkdir -p $O
python bench.py > $O/r02_${T}_bench_n1.json 2> $O/bench_err.log
tail -1 $O/r02_${T}_bench_n1.json | cut -c1-300
python bench.py --impl reference --steps 3 --warmup 1 > $O/r02_${T}_bench_reference_arm.json 2>> $O/bench_err.log
tail -1 $O/r02_${T}_bench_reference_arm.json | cut -c1-300
python tools/stage_times.py --tag C2 > $O/r02_${T}_stage_times.txt 2>&1
python tools/stage_times.py --scene inst --width 3840 --height 2160 --bounces 3 --passes 4 --tag C3 >> $O/r02_${T}_stage_times.txt 2>&1
python tools/stage_times.py --scene cornell --width 256 --height 256 --bounces 2 --flags 3 --tag C1 >> $O/r02_${T}_stage_times.txt 2>&1
cat $O/r02_${T}_stage_times.txt | cut -c1-240
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file $O/r02_${T}_launches.csv python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-extras > $O/ncu_bench.log 2>&1
timeout 900 ncu --set full --import-source on --clock-control none -k regex:"trace_kernel|k_gi_step|k_shade_primary|k_di_finish" -s 52 -c 13 -o $O/r02_${T}_pass -f python tools/prof_pass.py --passes 3 --opt PASS_PARTS=1 --opt PASS_PIPELINE=0 > $O/ncu_full.log 2>&1
tail -3 $O/ncu_full.log
RTX_B200_LIB=build/variants/timeline.so python tools/pass_timeline.py > $O/tl.txt 2>&1
python tools/pass_timeline.py --analyse $O/tl.txt > $O/r02_${T}_trace_timeline.txt
tail -5 $O/bench_err.log
ls -la $O | tail -20
