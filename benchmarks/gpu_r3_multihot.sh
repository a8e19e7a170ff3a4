#!/bin/bash
# Per-table pooling factors visit: build, the new multi-hot GPU tests, the existing kernels against a
# checkout of the parent commit (hotpath.py alternated in one session), benchmarks/multihot.py, the whole
# GPU suite, smoke() and bench.py for both builds.  $1 = a built checkout of the parent commit,
# $2 = the directory that receives the logs and JSON lines (created if missing).
PARENT=${1:?usage: gpu_r3_multihot.sh <built checkout of the parent commit> <output directory>}
O=${2:?usage: gpu_r3_multihot.sh <built checkout of the parent commit> <output directory>}
mkdir -p "$O"
PARENT=$(cd "$PARENT" && pwd); O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1 || { tail -30 $O/build.log; exit 1; }
timeout 900 python -m pytest tests/test_gpu_multihot.py -q -x -m gpu > $O/pytest_multihot.log 2>&1
for i in 1 2; do
  (cd $PARENT && python benchmarks/hotpath.py --workload terabyte --no-interaction) >> $O/hotpath_parent_terabyte.jsonl
  python benchmarks/hotpath.py --workload terabyte --no-interaction >> $O/hotpath_pr_terabyte.jsonl
  (cd $PARENT && python benchmarks/hotpath.py --workload kaggle --no-interaction) >> $O/hotpath_parent_kaggle.jsonl
  python benchmarks/hotpath.py --workload kaggle --no-interaction >> $O/hotpath_pr_kaggle.jsonl
done
timeout 1200 python benchmarks/multihot.py --mode ab full step --out $O/multihot.jsonl > $O/multihot.log 2>&1
timeout 1500 python -m pytest tests -q -m gpu > $O/pytest_gpu_all.log 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1
python bench.py --gpus 1 --steps 50 --warmup 10 > $O/bench.json
(cd $PARENT && python bench.py --gpus 1 --steps 50 --warmup 10) > $O/bench_parent.json
