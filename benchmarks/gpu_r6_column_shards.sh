#!/bin/bash
# Column-wise sharding visit, in stages (one GPU):
#   suite   build, the whole GPU suite, smoke(), one bench.py run
#   ab      the fused owner side against a checkout of the parent commit (the p2p lookup kernel now reads a
#           destination offset per table): sharded_multihot.py --mode owner alternated, and bench.py
#   owner   benchmarks/sharded_multihot.py --mode owner --plan column, then --mode step (which reports itself
#           unmeasured on fewer than two GPUs)
# $1 = stage, $2 = the directory that receives the logs and JSON lines (created if missing), $3 = a checkout
# of the parent commit (stage ab only; built here).
STAGE=${1:?usage: gpu_r6_column_shards.sh suite|ab|owner <output directory> [parent checkout]}
O=${2:?usage: gpu_r6_column_shards.sh suite|ab|owner <output directory> [parent checkout]}
mkdir -p "$O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_$STAGE.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $O/build_$STAGE.log 2>&1 || { tail -30 $O/build_$STAGE.log; exit 1; }
case $STAGE in
  suite)
    timeout 900 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu_all.log 2>&1
    tail -15 $O/pytest_gpu_all.log
    python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1
    tail -2 $O/smoke.log
    python bench.py --gpus 1 --steps 100 --warmup 10 > $O/bench.jsonl 2>&1
    tail -1 $O/bench.jsonl
    ;;
  ab)
    PARENT=$(cd "${3:?stage ab needs the parent checkout}" && pwd)
    (cd $PARENT && python -c "import __graft_entry__ as g; g.build()") > $O/build_parent.log 2>&1 || { tail -30 $O/build_parent.log; exit 1; }
    (cd $PARENT && timeout 200 python benchmarks/sharded_multihot.py --mode owner --repeats 3) >> $O/owner_parent.jsonl 2>> $O/owner_parent.log
    timeout 200 python benchmarks/sharded_multihot.py --mode owner --repeats 3 >> $O/owner_pr.jsonl 2>> $O/owner_pr.log
    for i in 1 2; do
      (cd $PARENT && python bench.py --gpus 1 --steps 100 --warmup 10) >> $O/bench_parent.jsonl
      python bench.py --gpus 1 --steps 100 --warmup 10 >> $O/bench_pr.jsonl
    done
    ;;
  owner)
    timeout 240 python benchmarks/sharded_multihot.py --mode owner --plan column --repeats 3 --out $O/column_shards_owner.jsonl > $O/column_shards_owner.log 2>&1
    tail -c 1500 $O/column_shards_owner.log
    python benchmarks/sharded_multihot.py --mode step > $O/column_shards_step.jsonl 2>&1
    cat $O/column_shards_step.jsonl
    ;;
esac
