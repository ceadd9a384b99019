#!/bin/bash
# Round 2, fifth GPU call: head conv with 32-byte patch rows (SWIZZLE_32B A operand); LDATI alignment fix.
set -u
export PYTHONUNBUFFERED=1
OUT=gpurun_out/r2e
mkdir -p "$OUT"
timeout 900 python -m pytest tests/test_gpu_unet.py tests/test_gpu_ldati.py tests/test_gpu_pipeline.py tests/test_gpu_torch_reference.py -m gpu -q -x 2>&1 | tail -30 > "$OUT/pytest_gpu.txt"
tail -6 "$OUT/pytest_gpu.txt"
timeout 120 python tools/layer_times.py 4 5 > "$OUT/layer_times_sw32.txt" 2>&1; head -4 "$OUT/layer_times_sw32.txt"; tail -1 "$OUT/layer_times_sw32.txt"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.txt" 2>&1; tail -2 "$OUT/smoke.txt"
timeout 300 python bench.py --headline-only > "$OUT/bench_headline.json" 2> "$OUT/bench.err"; tail -c 1500 "$OUT/bench_headline.json"
