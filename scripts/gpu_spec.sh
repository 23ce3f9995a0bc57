#!/bin/bash
# spec decoder: parity tests of the codec hook, K1 throughput per kind, bench without the decode / scan overlap.
TAG=${1:-spec}
OUT=gpurun_out/$TAG
mkdir -p $OUT
( timeout 600 python -m pytest tests/test_gpu_parity.py -m gpu -x -q -k "lz4 or golden or overlap or residency" ) > $OUT/pytest.log 2>&1
tail -5 $OUT/pytest.log
if grep -q "failed\|error\|Timeout" $OUT/pytest.log; then echo "SPEC TESTS FAILED"; grep -E "Error|assert" $OUT/pytest.log | head; exit 1; fi
( timeout 900 python scripts/decode_kinds.py --rows 200000000 --reps 3 ) > $OUT/kinds_200M.txt 2> $OUT/kinds_200M.err
cut -c1-60,150-260 $OUT/kinds_200M.txt
( DFDB_NO_OVERLAP=1 timeout 900 python scripts/decode_kinds.py --rows 1000000000 --reps 3 --cols ia ) > $OUT/kinds_1B.txt 2> $OUT/kinds_1B.err
cut -c1-60,150-260 $OUT/kinds_1B.txt
for V in "DFDB_NO_OVERLAP=1"; do
( env $V timeout 900 python bench.py --steps 10 --warmup 3 --no-e2e --no-variants ) > $OUT/bench_$V.json 2> $OUT/bench_$V.err
python - <<PY
import json
b=json.loads(open("$OUT/bench_$V.json").read().strip().splitlines()[-1])
print("$V", "value", round(b["value"]/1e9,2), "G rows/s  ms", round(b["ms_per_step"],3), "phases", b["phases_ms_per_step"], "verified", b["verified"]["ok"])
PY
done
