#!/bin/bash
# Round-3 evidence run (synchronised BatchNorm): GPU test suite (the two-rank tests run when >= 2 GPUs are visible),
# smoke, bench.py on 1 and 2 GPUs, and profiles/bench_dp_sync_bn.py for every world size in {2, 4, 8} the machine has.
# Usage: profiles/capture_r3.sh [OUT]; everything lands in OUT (a fresh temporary directory by default) and is then copied
# to profiles/r3/.  The records there come from a box with one B200: the two-rank synchronised-BatchNorm tests ran with
# both ranks on that GPU (LCN_RECORD_DIR keeps their per-rank JSON), and the multi-GPU benches did not run.
set -x
OUT=${1:-$(mktemp -d)}
mkdir -p $OUT
export LCN_RECORD_DIR=$OUT
nvidia-smi --query-gpu=index,name,power.limit --format=csv > $OUT/gpus.csv
NGPU=$(nvidia-smi -L | wc -l)
python __graft_entry__.py build > $OUT/build.log 2>&1; echo "build rc=$?"
timeout 1500 python -m pytest tests -q -m gpu -rs > $OUT/tests_gpu.log 2>&1; echo "tests rc=$?"
python __graft_entry__.py smoke > $OUT/smoke.log 2>&1; echo "smoke rc=$?"
python bench.py --gpus 1 --steps 100 --warmup 10 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
for w in 2 4 8; do
  [ "$w" -le "$NGPU" ] || continue
  timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node=$w --master-addr 127.0.0.1 --master-port 29541 \
      bench.py --gpus $w --steps 200 --warmup 10 --no-cpu-baseline --infer-poses 0 > $OUT/bench_n$w.json 2> $OUT/bench_n$w.err
  echo "bench n$w rc=$?"
  timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node=$w --master-addr 127.0.0.1 --master-port 29561 \
      profiles/bench_dp_sync_bn.py 200 5 > $OUT/bench_dp_sync_bn_n$w.json 2> $OUT/bench_dp_sync_bn_n$w.err
  echo "sync bench n$w rc=$?"
done
ls -la $OUT
