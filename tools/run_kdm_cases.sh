#!/bin/bash
# depth-merged halo kernel bring-up: every case in its own process
cd "$(dirname "$0")/.."
for c in kdm_n32 kdm_two_src_d16 kdm_n64_many kdm_128_in kdm_fullres kdm_s2_small kdm_s2_odd kdm_s2_128 kdm_s2_fullres; do
  timeout 180 python tools/conv_debug.py $c 2 2>&1 | grep -E "CASE|bad|m=|rror" | head -8
done
