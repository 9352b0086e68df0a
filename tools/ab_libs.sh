#!/bin/bash
# Same-box A/B of two builds of the library (KIRAG_B200_LIB): alternating runs of tools/probe_knobs.py.
# usage: tools/ab_libs.sh LIB_A LIB_B ROWS BATCHES [ROUNDS]
# PROBE_D sets the corpus width; with AB_SAVE set, each build saves its results (D, I) under $AB_SAVE/a and $AB_SAVE/b.
A=$1; B=$2; ROWS=$3; BATCHES=$4; ROUNDS=${5:-2}
for r in $(seq 1 $ROUNDS); do
  for tag in a b; do
    if [ $tag = a ]; then L=$A; else L=$B; fi
    echo "== round $r lib $tag $L"
    KIRAG_B200_LIB=$L PROBE_STEPS=${PROBE_STEPS:-20} PROBE_REPS=1 PROBE_SAVE=${AB_SAVE:+$AB_SAVE/$tag} \
      python tools/probe_knobs.py $ROWS $BATCHES "" 2>&1 | grep "^rep"
  done
done
