#!/bin/bash
# One GPU: main's library against this tree's, default bench line (python bench.py --steps 10), three runs each,
# alternating; the third run of each dumps its outputs and the dumps are compared bit for bit.
#   impdar_b200/libimpdar_b200_main.so   main's tree, built with python -m impdar_b200._build --out=...
#   impdar_b200/libimpdar_b200.so        this tree (python -m impdar_b200._build)
TAG=${1:-r03b}
O=${2:?usage: $0 TAG OUTDIR}; mkdir -p $O   # logs, bench lines and the dumped outputs go here
L=$PWD/impdar_b200
LOG=$O/${TAG}_kirch_tile_ab.txt
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $LOG
for rep in 1 2 3; do
  for v in main new; do
    lib=$L/libimpdar_b200.so; [ $v = main ] && lib=$L/libimpdar_b200_main.so
    dump=""; [ $rep = 3 ] && dump="--dump-outputs $O/dump_$v"
    IMPDAR_B200_LIB=$lib timeout 900 python bench.py --steps 10 $dump 2>/dev/null | tail -1 > $O/${TAG}_bench_${v}_$rep.json
    python - $O/${TAG}_bench_${v}_$rep.json $v $rep <<'EOF' | tee -a $LOG
import json, sys
d = json.loads(open(sys.argv[1]).read()); r = d["roofline"]; rec = d["records"]
print("%-4s run %s  ms/step %.2f  kernel %s %.2f ms  frac %.3f  stolt %.3f ms  config2 %.4f ms  parity %.2e  sm_mhz %s"
      % (sys.argv[2], sys.argv[3], d["ms_per_step"], r["kernel"], r["kernel_ms"], r["frac"],
         rec["stolt_65536x8192"]["ms_per_step"], rec["kirchhoff_4096x2048_per_gpu"]["ms_per_step"],
         d["parity"]["rel_l2"], d["clocks"]["sm_mhz"]))
EOF
  done
done
python - $O/dump_main $O/dump_new <<'EOF' | tee -a $LOG
import glob, os, sys
import numpy as np
for f in sorted(glob.glob(os.path.join(sys.argv[1], "*.npy"))):
    a, b = np.load(f), np.load(os.path.join(sys.argv[2], os.path.basename(f)))
    same = a.shape == b.shape and np.array_equal(a, b, equal_nan=True)
    print("bitwise %-36s %-14s %s" % (os.path.basename(f), a.shape, "EQUAL" if same else "DIFFERENT"))
EOF
rm -rf $O/dump_main $O/dump_new
