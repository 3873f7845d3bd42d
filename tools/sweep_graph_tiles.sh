#!/bin/bash
# Tile-shape sweep of the generated PLANAR graph kernel on the C4 voice graph (run under gpurun).
# A store-only graph (no input stream) uses every stage as a store buffer (wait depth STAGES-1).
for tf in 32 64; do for st in 2 3 4 5; do for w in 1 2 3 4; do
  echo -n "TF=$tf STAGES=$st WARPS=$w  "
  CPROC_GRAPH_TF=$tf CPROC_GRAPH_STAGES=$st CPROC_GRAPH_WARPS=$w timeout 120 python tools/prof_one.py gvoice 3 2>&1 | tail -1
done; done; done
echo -n "default  "; timeout 120 python tools/prof_one.py gvoice 3 2>&1 | tail -1
