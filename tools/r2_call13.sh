#!/bin/bash
# A/B on ONE box (box-to-box spread is larger than the effects): epilogue warps 8 / 16, head 9 / 6 taps.
# The 16-warp and 9-tap switches have since been removed from the library; only the default runs remain.
set -u
export PYTHONUNBUFFERED=1
OUT=gpurun_out/r2h
mkdir -p "$OUT"
timeout 600 python -m pytest tests/test_gpu_unet.py tests/test_gpu_pipeline.py -m gpu -q -x 2>&1 | tail -5 > "$OUT/pytest_gpu.txt"; tail -3 "$OUT/pytest_gpu.txt"
run() { name=$1; shift; env "$@" timeout 120 python tools/layer_times.py 4 8 > "$OUT/layer_times_$name.txt" 2>&1; echo "== $name: $(head -1 $OUT/layer_times_$name.txt)"; grep -E "head|encoders.0.conv2|decoders.2.conv2|decoders.3.conv2" "$OUT/layer_times_$name.txt"; }
run default V2CE_X=0
run default_again V2CE_X=0
