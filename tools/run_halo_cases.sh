#!/bin/bash
# halo-tile kernel bring-up: every case in its own process
cd "$(dirname "$0")/.."
for c in halo_64_64 halo_n32 halo_128_res halo_two_src halo_512 halo_768 halo_wide halo_many halo_fullres_slice; do
  timeout 180 python tools/conv_debug.py $c 1 2>&1 | grep -E "CASE|bad|m=|rror" | head -8
done
