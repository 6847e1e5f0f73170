#!/bin/bash
# compute-sanitizer over every kernel family (tools/sanitize_run.py), round 2
mkdir -p gpurun_out/r2
out=gpurun_out/r2/sanitizer_r02.txt
: > $out
for tool in memcheck racecheck; do
  echo "== compute-sanitizer --tool $tool" >> $out
  timeout 900 compute-sanitizer --tool $tool python tools/sanitize_run.py 2>&1 | grep -E "sanitize_run done|ERROR SUMMARY|RACECHECK SUMMARY|Invalid|hazard|Error" | head -12 >> $out
done
cat $out
