#!/bin/bash
# A/B of traversal variants / scheduling thresholds on the bench workload (run under gpurun)
mkdir -p gpurun_out
out=gpurun_out/ab_trace.txt
rm -f $out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm --format=csv,noheader >> $out
C3="--scene inst --width 3840 --height 2160 --bounces 3 --passes 4"
for v in build/variants/*.so; do
  RTX_B200_LIB=$v python tools/stage_times.py >> $out 2>&1
  RTX_B200_LIB=$v python tools/stage_times.py $C3 --tag C3_$v >> $out 2>&1
done
for s in ${SCHEDS:-0x000101 0x0c0808 0x0c0404 0x100808 0x080808 0x0c1010 0x100c0c 0x140808 0x0c0c08 0x0c080c 0x101010 0x180c0c}; do
  python tools/build_variant.py sched_$s -DRTX_SCHED_DEFAULT=$s >> $out 2>&1
  RTX_B200_LIB=build/variants/sched_$s.so python tools/stage_times.py --tag C2_$s >> $out 2>&1
  RTX_B200_LIB=build/variants/sched_$s.so python tools/stage_times.py $C3 --tag C3_$s >> $out 2>&1
done
cut -c1-130 $out
