#!/bin/bash
# Jagged-bags visit (one GPU): build, the whole GPU suite (tests/test_gpu_jagged.py first) and smoke() into
# r07_pytest_gpu.log, one bench.py line into r07_bench.jsonl, then benchmarks/jagged.py (const / var / mean) into
# r07_jagged_b200.jsonl: the names profiles/README.md indexes.  The SASS comparison with the parent commit needs no
# GPU: profiles/sass_diff.py on the parent's and this tree's lookup.o, sort.o and update.o.
# $1 = the directory that receives the files (created if missing).
O=${1:?usage: gpu_r7_jagged.sh <output directory>}
mkdir -p "$O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/r07_gpu.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $O/r07_build.log 2>&1 || { tail -30 $O/r07_build.log; exit 1; }
L=$O/r07_pytest_gpu.log
cat $O/r07_gpu.txt > $L
timeout 600 python -m pytest tests/test_gpu_jagged.py -q -m gpu -p no:cacheprovider >> $L 2>&1
timeout 1200 python -m pytest tests -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_jagged.py >> $L 2>&1
python -c "import __graft_entry__ as g; g.smoke()" >> $L 2>&1
grep -E "passed|failed|error|smoke ok" $L | tail -8
python bench.py --gpus 1 --steps 100 --warmup 10 > $O/r07_bench.jsonl 2> $O/r07_bench.log
tail -1 $O/r07_bench.jsonl
timeout 600 python benchmarks/jagged.py --out $O/r07_jagged_b200.jsonl > $O/r07_jagged.log 2>&1
tail -c 2500 $O/r07_jagged.log
