#!/bin/bash
# Round-2 evidence on ONE B200: sanitizer passes on the new paths, ncu --set full of the fused pcg! and
# projcg kernels (reports are reduced to CSV here: the .ncu-rep files are too large to bring back), and
# the launch list of the bench command.
set -x
OUT=gpurun_out
for tool in memcheck racecheck synccheck; do
  compute-sanitizer --tool $tool python tools/sanitize_small.py r2 > $OUT/r2_sanitizer_$tool.log 2>&1
  tail -3 $OUT/r2_sanitizer_$tool.log
done
ncu --set full --clock-control none -k regex:fused_pcg -s 1 -c 1 -o /tmp/r2_pcg python tools/c5_quick.py > $OUT/r2_ncu_pcg.log 2>&1
ncu -i /tmp/r2_pcg.ncu-rep --page details --csv > $OUT/r2_fused_pcg_details.csv 2>/dev/null
ncu -i /tmp/r2_pcg.ncu-rep --page raw --csv > $OUT/r2_fused_pcg_raw.csv 2>/dev/null
ncu --set full --clock-control none -k regex:fused_projcg -s 1 -c 1 -o /tmp/r2_projcg python tools/c5_quick.py > $OUT/r2_ncu_projcg.log 2>&1
ncu -i /tmp/r2_projcg.ncu-rep --page details --csv > $OUT/r2_fused_projcg_details.csv 2>/dev/null
ncu -i /tmp/r2_projcg.ncu-rep --page raw --csv > $OUT/r2_fused_projcg_raw.csv 2>/dev/null
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $OUT/r2_launches_bench.csv python bench.py --steps 2 --warmup 1 > $OUT/r2_bench_under_ncu.log 2>&1
ls -la $OUT | tail -20
