#!/bin/bash
# One GPU, three steps (each under ten minutes):
#   tests   : the GPU test suite and smoke()
#   lateral : scripts/bench_kirchhoff_lateral.py (layered tile / general against the two lateral paths, run-width sweep)
#   ab      : main's tree against this one with the default bench line (python bench.py --steps 10), alternating, two
#             runs each; the second run of each dumps its outputs and the dumps are compared bit for bit.  MAIN (default
#             _ab_main) is a built copy of main's whole tree.
WHAT=${1:?usage: $0 tests|lateral|ab TAG OUTDIR}
TAG=${2:-r06}
O=${3:?usage: $0 tests|lateral|ab TAG OUTDIR}; mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/${TAG}_${WHAT}_gpu.txt
if [ $WHAT = tests ]; then
  timeout 600 python -m pytest -q -m gpu tests/ -p no:cacheprovider 2>&1 | tail -40 > $O/${TAG}_gpu_tests.log
  tail -3 $O/${TAG}_gpu_tests.log
  timeout 100 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 > $O/${TAG}_smoke.log
  cat $O/${TAG}_smoke.log
elif [ $WHAT = lateral ]; then
  timeout 580 python scripts/bench_kirchhoff_lateral.py --steps 10 --warmup 3 > $O/bench_kirchhoff_lateral_${TAG}.log 2>&1
  tail -1 $O/bench_kirchhoff_lateral_${TAG}.log > $O/bench_kirchhoff_lateral_${TAG}.json
  tail -5 $O/bench_kirchhoff_lateral_${TAG}.log
else
  MAIN=${MAIN:-_ab_main}
  OUT=$PWD/$O
  LOG=$OUT/${TAG}_ab.txt
  cp $OUT/${TAG}_${WHAT}_gpu.txt $LOG
  for rep in 1 2; do
    for v in main new; do
      dir=$PWD; [ $v = main ] && dir=$PWD/$MAIN
      dump=""; [ $rep = 2 ] && dump="--dump-outputs $OUT/dump_$v"
      (cd $dir && timeout 150 python bench.py --steps 10 $dump 2>/dev/null | tail -1) > $OUT/${TAG}_bench_${v}_$rep.json
      python scripts/ab_line.py $OUT/${TAG}_bench_${v}_$rep.json $v $rep | tee -a $LOG
    done
  done
  python scripts/ab_line.py --compare $OUT/dump_main $OUT/dump_new | tee -a $LOG
  rm -rf $OUT/dump_main $OUT/dump_new
fi
