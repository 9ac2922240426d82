#!/bin/bash
# compute-sanitizer over scripts/sanitize_target.py: memcheck, racecheck (shared-memory hazards; the LK kernels reuse shared
# scratch across named barriers), synccheck, initcheck.  usage (under gpurun): bash scripts/gpu_sanitize.sh <tag>
OUT=gpurun_out/${1:-r02_sanitize}
mkdir -p $OUT
python scripts/sanitize_target.py > $OUT/plain.log 2>&1; echo "plain run exit $?" | tee -a $OUT/plain.log
for tool in memcheck racecheck synccheck initcheck; do
  log=$OUT/${tool}.log
  timeout 1500 compute-sanitizer --tool $tool --print-limit 20 python scripts/sanitize_target.py > $log 2>&1
  echo "$tool exit $?: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|sanitize_target:' $log | tr '\n' ' ')"
done | tee $OUT/summary.txt
