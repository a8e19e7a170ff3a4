#!/bin/bash
# Mixed-P table-sharded visit, in stages (one GPU):
#   suite   build, the whole GPU suite, smoke()
#   ab      the uniform path against a checkout of the parent commit: hotpath.py and bench.py alternated
#   owner   benchmarks/sharded_multihot.py --mode owner, then --mode step (which reports itself unmeasured
#           on fewer than two GPUs)
# $1 = stage, $2 = the directory that receives the logs and JSON lines (created if missing), $3 = a checkout
# of the parent commit (stage ab only; built here).
STAGE=${1:?usage: gpu_r4_sharded_multihot.sh suite|ab|owner <output directory> [parent checkout]}
O=${2:?usage: gpu_r4_sharded_multihot.sh suite|ab|owner <output directory> [parent checkout]}
mkdir -p "$O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_$STAGE.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $O/build_$STAGE.log 2>&1 || { tail -30 $O/build_$STAGE.log; exit 1; }
case $STAGE in
  suite)
    timeout 480 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu_all.log 2>&1
    tail -3 $O/pytest_gpu_all.log
    python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1
    tail -2 $O/smoke.log
    ;;
  ab)
    PARENT=$(cd "${3:?stage ab needs the parent checkout}" && pwd)
    (cd $PARENT && python -c "import __graft_entry__ as g; g.build()") > $O/build_parent.log 2>&1 || { tail -30 $O/build_parent.log; exit 1; }
    for i in 1 2; do
      (cd $PARENT && python benchmarks/hotpath.py --workload terabyte --no-interaction) >> $O/hotpath_parent_terabyte.jsonl
      python benchmarks/hotpath.py --workload terabyte --no-interaction >> $O/hotpath_pr_terabyte.jsonl
      (cd $PARENT && python bench.py --gpus 1 --steps 100 --warmup 10) >> $O/bench_parent.jsonl
      python bench.py --gpus 1 --steps 100 --warmup 10 >> $O/bench_pr.jsonl
    done
    (cd $PARENT && python benchmarks/hotpath.py --workload kaggle --no-interaction) >> $O/hotpath_parent_kaggle.jsonl
    python benchmarks/hotpath.py --workload kaggle --no-interaction >> $O/hotpath_pr_kaggle.jsonl
    ;;
  owner)
    timeout 420 python benchmarks/sharded_multihot.py --mode owner --out $O/sharded_multihot_owner.jsonl > $O/sharded_multihot_owner.log 2>&1
    tail -c 600 $O/sharded_multihot_owner.log
    python benchmarks/sharded_multihot.py --mode step > $O/sharded_multihot_step.jsonl 2>&1
    cat $O/sharded_multihot_step.jsonl
    ;;
esac
