#!/bin/bash
# Uniform entry points served by the per-table-pooling kernels: this tree against a checkout of the parent
# commit, alternated in one session (one GPU).  $1 = the directory that receives the logs and JSON lines
# (created if missing), $2 = the parent checkout, already built.
O=${1:?usage: gpu_r5_uniform_via_mp.sh <output directory> <parent checkout>}
PARENT=$(cd "${2:?usage: gpu_r5_uniform_via_mp.sh <output directory> <parent checkout>}" && pwd)
mkdir -p "$O"
O=$(cd "$O" && pwd)
ME=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu.txt 2>&1
# bench.py: samples/s and the outputs of the last timed step, which must be byte-identical between builds
for i in 1 2; do
  for w in terabyte kaggle; do
    for b in parent pr; do
      d=$ME; [ $b = parent ] && d=$PARENT
      (cd $d && python bench.py --gpus 1 --steps 100 --warmup 10 --workload $w --no-cpu-baseline --no-host-leg \
         --dump-outputs $O/dump_${w}_${b}_$i) 2> $O/bench_${w}_${b}_$i.log | tail -1 \
        | sed "s/^/{\"build\": \"$b\", \"line\": /; s/\$/}/" >> $O/bench_ab.jsonl
    done
    for f in $(cd $O/dump_${w}_pr_$i && ls); do
      cmp -s $O/dump_${w}_parent_$i/$f $O/dump_${w}_pr_$i/$f && echo "$w run $i $f identical" || echo "$w run $i $f DIFFERENT"
    done >> $O/dump_compare.txt
  done
done
# embedding kernels alone: Terabyte B 2048 / 16384, Kaggle, and one radix-sort case (L = 32768 per table)
for i in 1 2; do
  for b in parent pr; do
    d=$ME; [ $b = parent ] && d=$PARENT
    (cd $d && python benchmarks/hotpath.py --workload terabyte --D 128 --B 2048 --no-interaction) >> $O/hotpath_${b}.jsonl
    (cd $d && python benchmarks/hotpath.py --workload terabyte --D 128 --B 16384 --no-interaction) >> $O/hotpath_${b}.jsonl
    (cd $d && python benchmarks/hotpath.py --workload kaggle --no-interaction) >> $O/hotpath_${b}.jsonl
    (cd $d && python benchmarks/hotpath.py --rows 10000000 --D 128 --B 2048 --P 16 --no-interaction) >> $O/hotpath_${b}.jsonl
  done
done
python benchmarks/multihot.py --mode full --out $O/multihot_full.jsonl > $O/multihot_full.log 2>&1
