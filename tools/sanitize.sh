#!/bin/bash
# compute-sanitizer over every kernel family of the library on small shapes (run under gpurun, 1 GPU).
# The plain run comes first and must pass; each tool then gets its own bounded run.  Logs go to gpurun_out/ and
# the summaries are copied to profiles/ by hand.
set -u
OUT=gpurun_out
mkdir -p $OUT
nvcc -O2 -std=c++17 -o $OUT/sanitize_driver tools/sanitize_driver.cu -Lkirag_b200 -lkirag_b200 -Xlinker -rpath -Xlinker $PWD/kirag_b200 || exit 1
$OUT/sanitize_driver all > $OUT/r2_sanitize_plain.log 2>&1
echo "plain rc=$?"; tail -3 $OUT/r2_sanitize_plain.log
for tool in memcheck racecheck synccheck initcheck; do
  for c in scan search pool exchange topk host_rescore host_exact multi_merge remove_compact id_map; do
    timeout 900 compute-sanitizer --tool $tool --error-exitcode 9 --print-limit 20 $OUT/sanitize_driver $c > $OUT/r2_sanitize_${tool}_$c.log 2>&1
    rc=$?
    echo "$tool $c rc=$rc: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|passed' $OUT/r2_sanitize_${tool}_$c.log | tr '\n' ' ')"
  done
done
