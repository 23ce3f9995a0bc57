#!/bin/bash
# A/B: decoder flavours on the nullable / grid columns.
OUT=gpurun_out/${1:-ab2}
mkdir -p $OUT
( timeout 600 python -m pytest tests/test_gpu_parity.py -m gpu -x -q -k "lz4 or codec" ) > $OUT/pytest.log 2>&1
tail -2 $OUT/pytest.log
for F in 0 2 4; do
echo "flavour $F"
( DFDB_LZ4_FLAVOUR=$F timeout 600 python scripts/decode_kinds.py --rows 200000000 --reps 3 --cols ma,mb,fg,sq ) > $OUT/kinds_f$F.txt 2> $OUT/kinds_f$F.err
cut -c1-60,150-260 $OUT/kinds_f$F.txt
done
