#!/bin/bash
# spec decoder iteration: codec parity tests, bench, ncu capture with source page, K1 per kind.
TAG=${1:-spec2}
OUT=gpurun_out/$TAG
mkdir -p $OUT
( timeout 900 python -m pytest tests/test_gpu_parity.py -m gpu -x -q -k "lz4 or golden or overlap or residency or filter_aggregate or codec" ) > $OUT/pytest.log 2>&1
tail -3 $OUT/pytest.log
if grep -q "failed\|error\|Timeout" $OUT/pytest.log; then echo "SPEC TESTS FAILED"; grep -E "Error|assert" $OUT/pytest.log | head; exit 1; fi
for V in "DFDB_NO_OVERLAP=1" $EXTRA_VARIANTS; do
( env ${V//,/ } timeout 900 python bench.py --steps 10 --warmup 3 --no-e2e --no-variants ) > $OUT/bench_$V.json 2> $OUT/bench_$V.err
python - <<PY
import json
b=json.loads(open("$OUT/bench_$V.json").read().strip().splitlines()[-1])
print("$V", "value", round(b["value"]/1e9,2), "G rows/s  ms", round(b["ms_per_step"],3), "phases", b["phases_ms_per_step"], "kernel", b["roofline"]["kernel"], "frac", round(b["roofline"]["frac"],3), "verified", b["verified"]["ok"])
PY
done
if [ -z "$NO_NCU" ]; then
DFDB_NO_OVERLAP=1 timeout 900 ncu --set full --clock-control none --import-source on -k regex:lz4_decode_spec -s 2 -c 1 -o $OUT/cap python bench.py --steps 2 --warmup 1 --no-e2e --no-variants --no-verify > $OUT/ncu.log 2>&1
tail -2 $OUT/ncu.log
ncu -i $OUT/cap.ncu-rep --page details > $OUT/details.txt 2>/dev/null
ncu -i $OUT/cap.ncu-rep --page raw --csv > $OUT/raw.csv 2>/dev/null
ncu -i $OUT/cap.ncu-rep --page source --csv --print-source cuda,sass > $OUT/source.csv 2>/dev/null
rm -f $OUT/cap.ncu-rep
grep -E "Duration|Executed Ipc|Issue Slots Busy|Registers Per|Achieved Occupancy|DRAM Throughput|Executed Instructions  " $OUT/details.txt | head -20
fi
if [ -z "$NO_KINDS" ]; then
( timeout 900 python scripts/decode_kinds.py --rows 200000000 --reps 3 ) > $OUT/kinds_200M.txt 2> $OUT/kinds_200M.err
cut -c1-60,150-260 $OUT/kinds_200M.txt
fi
