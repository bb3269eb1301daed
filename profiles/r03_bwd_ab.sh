#!/bin/bash
# A/B of the blend backward on one GPU: the parent commit's library against this tree's, alternating run by run.
#   log_b200/_lib/ab/old.so   built from the parent commit (same nvcc flags as log_b200/build.py)
#   log_b200/_lib/ab/new.so   this tree's library
#   log_b200/_lib/ab/sg.so    (optional) the fallback measured while this change was developed: per-splat shared
#                             accumulators kept, their CAS-loop adds spread over the 4 lanes of a group (3 add sites)
# Each is copied over log_b200/_lib/liblog_b200_raster.so in turn; new.so is put back at the end.
# Everything is written under OUT_DIR.  Then: --dump-outputs of old and new at 10 M (compared by profiles/r03_compare_dumps.py), smoke() and the GPU suite.
set -u
OUT=${1:?usage: profiles/r03_bwd_ab.sh OUT_DIR}
REPS=${REPS:-3}
LIB=log_b200/_lib/liblog_b200_raster.so
AB=log_b200/_lib/ab
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv > $OUT/gpu.csv 2>&1
VARIANTS="old new"
[ -f $AB/sg.so ] && VARIANTS="old new sg"

run() {      # run <variant> <workload> <rep> <steps>
  cp $AB/$1.so $LIB
  timeout 600 python bench.py --gpus 1 --workload $2 --steps $4 --warmup 5 --no-e2e --no-cpu-baseline \
    > $OUT/bench_$2_$1_$3.json 2> $OUT/bench_$2_$1_$3.err
}
for rep in $(seq 1 $REPS); do
  for v in $VARIANTS; do run $v 10m $rep 20; done
  for v in $VARIANTS; do run $v 100k $rep 50; done
  for v in $VARIANTS; do run $v big300k $rep 20; done
done
for v in old new; do
  cp $AB/$v.so $LIB
  timeout 600 python bench.py --gpus 1 --steps 3 --warmup 3 --no-e2e --no-cpu-baseline --dump-outputs $OUT/dump_$v \
    > $OUT/dump_$v.json 2> $OUT/dump_$v.err
done
cp $AB/new.so $LIB
python profiles/r03_compare_dumps.py $OUT/dump_old $OUT/dump_new > $OUT/compare_dumps.txt 2>&1
timeout 300 python -c "import __graft_entry__ as e; e.smoke()" > $OUT/smoke.log 2>&1
echo "smoke rc=$?" > $OUT/summary.txt
timeout 1200 python -m pytest tests -q -m gpu -p no:cacheprovider > $OUT/gpu_suite.log 2>&1
echo "gpu suite rc=$?" >> $OUT/summary.txt
python profiles/r03_ab_table.py $OUT > $OUT/table.md 2>&1
cat $OUT/gpu.csv $OUT/table.md $OUT/compare_dumps.txt $OUT/summary.txt
tail -n 3 $OUT/gpu_suite.log
