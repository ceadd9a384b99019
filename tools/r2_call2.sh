#!/bin/bash
# Round 2, second GPU call: one-sweep LDATI sort + quad-dealt emit + fused count/event-frame sums + 4-launch select.
set -u
export PYTHONUNBUFFERED=1
OUT=gpurun_out/r2b
mkdir -p "$OUT"
timeout 900 python -m pytest tests -m gpu -q 2>&1 | tail -60 > "$OUT/pytest_gpu.txt"
tail -8 "$OUT/pytest_gpu.txt"
timeout 300 python tools/ldati_bench.py 5 --table > "$OUT/ldati_table.json" 2> "$OUT/ldati_table.err"
python -c "
import json
d=json.load(open('$OUT/ldati_table.json'))
for k,v in d.items(): print(k, round(v['ms'],3), 'ms', round(v['frac_of_hbm_peak'],3))
"
for d in rand randint10 sparse; do
  timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file "$OUT/ldati_launches_$d.csv" \
      python tools/ldati_bench.py 1 --pairs 24 --dist $d > "$OUT/ldati_$d.log" 2>&1
done
timeout 300 ncu --set full --clock-control none --import-source on -k regex:'emit_kernel|osw_scatter_kernel|osw_hist_kernel|pack_kernel' \
    -s 5 -c 5 -o "$OUT/ldati_full_rand" python tools/ldati_bench.py 1 --pairs 24 --dist rand > "$OUT/ncu_ldati_rand.log" 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:'emit_kernel' \
    -s 1 -c 1 -o "$OUT/emit_full_randint" python tools/ldati_bench.py 1 --pairs 24 --dist randint10 > "$OUT/ncu_emit_randint.log" 2>&1
timeout 420 python bench.py > "$OUT/bench.json" 2> "$OUT/bench.err"
tail -c 300 "$OUT/bench.json"; tail -3 "$OUT/bench.err"
ls -la "$OUT"
