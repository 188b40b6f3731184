#!/bin/bash
# One GPU: tile-kernel consumer variants against main's library on the headline, alternating; outputs bit for bit.
#   impdar_b200/libimpdar_b200_main.so   main's tree, built with python -m impdar_b200._build --out=...
#   impdar_b200/libimpdar_b200.so        the decoded walk as the compiler unrolls it by default (4x)
#   impdar_b200/libimpdar_b200_u{1,2}.so the same with `#pragma unroll 1` / `2` on the walk loop
# The plain loop (u1) measured fastest and is what kirchhoff_tile.cuh now holds; the other two were built from the
# same source with the pragma changed.
TAG=${1:-r03a}
O=${2:?usage: $0 TAG OUTDIR}; mkdir -p $O   # logs, bench lines and the dumped outputs go here
L=$PWD/impdar_b200
LOG=$O/${TAG}_kirch_tile_variants.txt
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $LOG
quick() {   # $1 = label, $2 = library
  IMPDAR_B200_LIB=$2 timeout 600 python bench.py --steps 5 --warmup 2 --no-cpu-baseline --no-e2e --no-parity --no-records \
    2>/dev/null | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read()); r=d['roofline']
print('%-5s ms/step %.2f kernel %s %.2f ms frac %.3f sm_mhz %s' % ('$1', d['ms_per_step'], r['kernel'], r['kernel_ms_per_step'], r['frac'], d['clocks']['sm_mhz']))" | tee -a $LOG
}
for rep in 1 2; do
  quick main $L/libimpdar_b200_main.so
  quick new $L/libimpdar_b200.so
  quick u1 $L/libimpdar_b200_u1.so
  quick u2 $L/libimpdar_b200_u2.so
done
for v in main new; do
  lib=$L/libimpdar_b200.so; [ $v = main ] && lib=$L/libimpdar_b200_main.so
  IMPDAR_B200_LIB=$lib timeout 900 python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-e2e --dump-outputs $O/dump_$v \
    2>/dev/null | tail -1 > $O/${TAG}_bench_dump_$v.json
done
python - <<EOF | tee -a $LOG
import glob, os, numpy as np
for f in sorted(glob.glob("$O/dump_main/*.npy")):
    a = np.load(f); b = np.load(os.path.join("$O/dump_new", os.path.basename(f)))
    print("bitwise %-40s %s %s" % (os.path.basename(f), a.shape, "EQUAL" if np.array_equal(a, b, equal_nan=True) else "DIFFERENT (max abs %.3e)" % np.nanmax(np.abs(a - b))))
EOF
rm -rf $O/dump_main $O/dump_new
