#!/bin/bash
# Weighted-bags visit (one GPU): build, the whole GPU suite (tests/test_gpu_jagged_weighted.py first) and smoke() into
# r08_pytest_gpu.log, one bench.py line into r08_bench.jsonl, then benchmarks/jagged.py (var / weighted) into
# r08_weighted_b200.jsonl: the names profiles/README.md indexes.  The SASS comparison with the parent commit needs no
# GPU: profiles/sass_diff.py on the parent's and this tree's lookup.o, sort.o and update.o.
# $1 = the directory that receives the files (created if missing).
O=${1:?usage: gpu_r8_weighted.sh <output directory>}
mkdir -p "$O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/r08_gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $O/r08_build.log 2>&1 || { tail -30 $O/r08_build.log; exit 1; }
L=$O/r08_pytest_gpu.log
cat $O/r08_gpu.txt > $L
timeout 600 python -m pytest tests/test_gpu_jagged_weighted.py -q -m gpu -p no:cacheprovider >> $L 2>&1
timeout 1200 python -m pytest tests -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_jagged_weighted.py >> $L 2>&1
python -c "import __graft_entry__ as g; g.smoke()" >> $L 2>&1
grep -E "passed|failed|error|smoke ok" $L | tail -8
python bench.py --gpus 1 --steps 100 --warmup 10 > $O/r08_bench.jsonl 2> $O/r08_bench.log
tail -1 $O/r08_bench.jsonl
timeout 600 python benchmarks/jagged.py --mode var weighted --out $O/r08_weighted_b200.jsonl > $O/r08_weighted.log 2>&1
tail -c 3000 $O/r08_weighted.log
