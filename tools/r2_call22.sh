#!/bin/bash
# A/B on ONE box: N tile 128 instead of 256 for the 256- / 512-channel halo layers (wave quantisation: 448 items = 3.03 waves).
# The N-tile switches have since been removed from the library (256-channel layers use 128); only the default runs remain.
set -u
export PYTHONUNBUFFERED=1
OUT=gpurun_out/r2l
mkdir -p "$OUT"
run() { name=$1; shift; env "$@" timeout 120 python tools/layer_times.py 4 8 > "$OUT/layer_times_$name.txt" 2>&1; echo "== $name: $(head -1 $OUT/layer_times_$name.txt) | $(tail -1 $OUT/layer_times_$name.txt)"; }
run default V2CE_X=0
run default_again V2CE_X=0
