#!/bin/bash
# compute-sanitizer evidence (memcheck / racecheck / synccheck) over one small launch of every kernel family.
# usage: tools/gpu_sanitize.sh [tag]   -> gpurun_out/sanitize_<tool>_<tag>.log (+ one-line summaries on stdout)
# FAMILIES="mc ..." limits the run to those kernel families of tools/sanitize.py (default: all of them)
tag=${1:-r02}
mkdir -p gpurun_out
for tool in memcheck racecheck synccheck; do
  for fam in ${FAMILIES:-generic fast ws direct tma dtma cluster pool aux mc}; do
    timeout 420 compute-sanitizer --tool $tool --print-limit 20 python tools/sanitize.py $fam \
        > gpurun_out/sanitize_${tool}_${fam}_${tag}.log 2>&1
    echo "$tool $fam rc=$? $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY' gpurun_out/sanitize_${tool}_${fam}_${tag}.log | tail -1)"
  done
done
