#!/bin/bash
# compute-sanitizer passes over tools/sanitize_driver.py on the GPU box; logs -> gpurun_out/
mkdir -p gpurun_out
for tool in memcheck racecheck synccheck initcheck; do
  timeout 600 compute-sanitizer --tool $tool --print-limit 20 python tools/sanitize_driver.py > gpurun_out/sanitize_$tool.log 2>&1
  echo "$tool rc=$? : $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|sanitize driver ok' gpurun_out/sanitize_$tool.log | tr '\n' ' ')"
done
