#!/bin/bash
# Sharded jagged-bags visit (one GPU): build, the whole GPU suite (tests/test_gpu_sharded_jagged.py first) and smoke()
# into r09_pytest_gpu.log, one bench.py line into r09_bench.jsonl, then benchmarks/sharded_jagged.py --mode owner into
# r09_sharded_jagged_owner.jsonl and --mode step into r09_sharded_jagged_step.jsonl: the names profiles/README.md
# indexes.  The SASS comparison with the parent commit needs no GPU: profiles/sass_diff.py on the parent's and this
# tree's lookup.o, sort.o, update.o and p2p.o.
# $1 = the directory that receives the files (created if missing).
O=${1:?usage: gpu_r9_sharded_jagged.sh <output directory>}
mkdir -p "$O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/r09_gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $O/r09_build.log 2>&1 || { tail -30 $O/r09_build.log; exit 1; }
L=$O/r09_pytest_gpu.log
cat $O/r09_gpu.txt > $L
timeout 900 python -m pytest tests/test_gpu_sharded_jagged.py -q -m gpu -p no:cacheprovider >> $L 2>&1
timeout 1200 python -m pytest tests -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_sharded_jagged.py >> $L 2>&1
python -c "import __graft_entry__ as g; g.smoke()" >> $L 2>&1
grep -E "passed|failed|error|smoke ok" $L | tail -8
python bench.py --gpus 1 --steps 100 --warmup 10 > $O/r09_bench.jsonl 2> $O/r09_bench.log
tail -1 $O/r09_bench.jsonl
timeout 900 python benchmarks/sharded_jagged.py --mode owner --out $O/r09_sharded_jagged_owner.jsonl > $O/r09_sharded_jagged.log 2>&1
python benchmarks/sharded_jagged.py --mode step > $O/r09_sharded_jagged_step.jsonl 2>> $O/r09_sharded_jagged.log
tail -c 2500 $O/r09_sharded_jagged.log
