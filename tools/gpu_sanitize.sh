#!/bin/bash
# compute-sanitizer (memcheck, racecheck, synccheck) over every kernel path at small sizes; summary -> gpurun_out/sanitizer_r02.txt
mkdir -p gpurun_out
OUT=gpurun_out/sanitizer_r02.txt
echo "# compute-sanitizer $(compute-sanitizer --version | head -1) on $(nvidia-smi --query-gpu=name --format=csv,noheader | head -1); cases = tools/sanitize_case.py" > $OUT
for tool in memcheck racecheck synccheck; do
  for c in thread warp radix slab3 strict io; do
    timeout 600 compute-sanitizer --tool $tool --print-limit 5 python tools/sanitize_case.py $c > gpurun_out/san_${tool}_$c.log 2>&1
    rc=$?
    summary=$(grep -E "ERROR SUMMARY|RACECHECK SUMMARY" gpurun_out/san_${tool}_$c.log | tail -1)
    okline=$(grep -E "^$c ok" gpurun_out/san_${tool}_$c.log | tail -1)
    echo "$tool $c: exit $rc | ${okline:-NO-OK-LINE} | ${summary:-no summary line}" | tee -a $OUT
  done
done
