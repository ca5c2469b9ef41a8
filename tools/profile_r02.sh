#!/bin/bash
# Round-2 profiling pass, run under gpurun on ONE GPU:   bash tools/profile_r02.sh [tag]
#  1. launch lists (ncu --metrics gpu__time_duration.sum) of `bench.py --config cN` -> gpurun_out/<tag>_launches_cN.csv
#  2. one `ncu --set full` capture of each config's dominant kernel(s)            -> gpurun_out/<tag>_full_cN.ncu-rep
# Numbers printed by runs under ncu are never bench values.
TAG=${1:-r02}
CONFIGS=${2:-"c1 c2 c3 c4 c5"}   # optional: only these configs
mkdir -p gpurun_out
B="python bench.py --steps 2 --warmup 3 --no-e2e --no-cpu-baseline"
for c in $CONFIGS; do
  L=""; [ $c = c5 ] && L="--lines 2097152"
  timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv \
      --log-file gpurun_out/${TAG}_launches_$c.csv $B --config $c $L > gpurun_out/${TAG}_launches_$c.log 2>&1
done
declare -A K=( [c1]="split_mask_kernel|split_scan_kernel|split_emit_kernel" [c2]="regex_tdfa" [c3]="split_mask_kernel|split_scan_kernel|split_emit_kernel|ml_pass_kernel|ml_tile_scan_kernel" [c4]="delim_tiled_kernel|regex_tdfa_staged" [c5]="regex_tdfa_multi" )
declare -A NK=( [c1]=3 [c2]=2 [c3]=8 [c4]=2 [c5]=2 )
declare -A SK=( [c1]=9 [c2]=4 [c3]=24 [c4]=6 [c5]=4 )
for c in $CONFIGS; do
  L=""; [ $c = c5 ] && L="--lines 1048576"
  timeout 900 ncu --set full --clock-control none --import-source on -k "regex:${K[$c]}" -s ${SK[$c]} -c ${NK[$c]} -f \
      -o gpurun_out/${TAG}_full_$c $B --config $c $L > gpurun_out/${TAG}_full_$c.log 2>&1
  # the summaries travel back (gpurun_out is capped at 64 MiB); only the headline config's capture is kept whole
  python profiles/summarize.py gpurun_out/${TAG}_full_$c.ncu-rep "" ${TAG}_full_$c gpurun_out >> gpurun_out/${TAG}_full_$c.log 2>&1
  [ $c = c2 ] || rm -f gpurun_out/${TAG}_full_$c.ncu-rep
done
ls -la gpurun_out/${TAG}_*
