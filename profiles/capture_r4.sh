#!/bin/bash
# Round-4 evidence run (backward BatchNorm kernels sized to run beside the weight-gradient GEMM): bench.py at config 2
# against the parent commit, alternated three times, configs 4 and 5 twice each, the start-to-start step timeline of
# both (profiling builds), --dump-outputs three times on the parent and once here (compared by profiles/compare_dumps.py), the
# GPU test suite and smoke.
# Usage: profiles/capture_r4.sh OUT PARENT -- PARENT is a checkout of the parent commit with both of its libraries built
# (make, make prof in lcn_pose_b200/csrc); everything lands in OUT and is then copied to profiles/r4/.
set -x
mkdir -p "$1"
OUT=$(cd "$1" && pwd)
PARENT=$2
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm --format=csv > $OUT/gpus.csv
python __graft_entry__.py build > $OUT/build.log 2>&1; echo "build rc=$?"
make -C lcn_pose_b200/csrc -j8 prof >> $OUT/build.log 2>&1; echo "prof build rc=$?"
BENCH="bench.py --gpus 1 --warmup 10 --no-cpu-baseline --infer-poses 0"
for i in 1 2 3; do
  (cd $PARENT && python $BENCH --steps 200) > $OUT/bench_parent_$i.json 2> $OUT/bench_parent_$i.err
  python $BENCH --steps 200 > $OUT/bench_$i.json 2> $OUT/bench_$i.err
done
for c in 4 5; do
  for i in 1 2; do
    (cd $PARENT && timeout 300 python $BENCH --steps 100 --config $c) > $OUT/bench_parent_config${c}_$i.json 2> $OUT/bench_parent_config${c}_$i.err
    timeout 300 python $BENCH --steps 100 --config $c > $OUT/bench_config${c}_$i.json 2> $OUT/bench_config${c}_$i.err
  done
done
{ set +x; } 2> /dev/null      # the logs hold the timelines only
(cd $PARENT && LCN_B200_LIB=lcn_pose_b200/liblcn_b200_prof.so python profiles/ktrace_step.py) > $OUT/ktrace_step_parent.log 2>&1
LCN_B200_LIB=lcn_pose_b200/liblcn_b200_prof.so python profiles/ktrace_step.py > $OUT/ktrace_step.log 2>&1
set -x
D=$(mktemp -d)
for i in 1 2 3; do
  (cd $PARENT && python $BENCH --steps 20 --dump-outputs $D/parent_$i) > /dev/null 2>&1; echo "dump parent $i rc=$?"
done
python $BENCH --steps 20 --dump-outputs $D/branch > /dev/null 2>&1; echo "dump rc=$?"
{ python profiles/compare_dumps.py $D/parent_1 $D/parent_2 parent1-vs-parent2
  python profiles/compare_dumps.py $D/parent_1 $D/parent_3 parent1-vs-parent3
  python profiles/compare_dumps.py $D/parent_2 $D/parent_3 parent2-vs-parent3
  for i in 1 2 3; do python profiles/compare_dumps.py $D/parent_$i $D/branch branch-vs-parent$i; done; } > $OUT/dump_compare.jsonl
rm -rf $D
timeout 1500 python -m pytest tests -q -m gpu -rs > $OUT/tests_gpu.log 2>&1; echo "tests rc=$?"
python __graft_entry__.py smoke > $OUT/smoke.log 2>&1; echo "smoke rc=$?"
ls -la $OUT
