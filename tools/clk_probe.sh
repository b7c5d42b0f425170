#!/bin/bash
# usage: clk_probe.sh <tag> <B> <reps>   (tag names the output file clk_<tag>.csv)
nvidia-smi --query-gpu=clocks.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.sw_power_cap,clocks_event_reasons.hw_slowdown,clocks_event_reasons.sw_thermal_slowdown,temperature.gpu --format=csv,noheader -lms 100 > gpurun_out/clk_$1.csv &
SMI=$!
python tools/k2_probe.py $2 $3
kill $SMI
sort gpurun_out/clk_$1.csv | uniq -c | sort -rn | head -8
