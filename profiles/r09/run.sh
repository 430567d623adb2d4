#!/bin/bash
# Round 9: the unchanged shapes (L <= 64) against the parent commit on one GPU, in one session:
#   profiles/r09/run.sh <parent tree, built> <output directory>
# 1. bench.py on c3 (default), c4 and c5, alternating the parent tree and this one (old, new, new, old, old, new);
# 2. scripts/ab_outputs.py in both trees (L <= 64 shapes of every path and projection kernel), digests compared.
# The wide-model benchmark runs on its own: python scripts/bench_wide.py --out <dir>/bench_wide.jsonl
old=$1; out=$2
mkdir -p $out
here=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv,noheader | head -1 | tee $out/card.txt
for wl in c3 c4 c5; do
  run=0
  for b in old new new old old new; do
    run=$((run + 1))
    if [ $b = old ]; then cd $old; else cd $here; fi
    python bench.py --gpus 1 --workload $wl --no-cpu --no-also --no-e2e > $here/$out/bench_${wl}_${run}_$b.json 2> $here/$out/bench_${wl}_${run}_$b.err
    cd $here
  done
done
(cd $old && python scripts/ab_outputs.py $here/$out/ab_outputs_old.json) > $out/ab_outputs.log 2>&1
python scripts/ab_outputs.py $out/ab_outputs_new.json >> $out/ab_outputs.log 2>&1
python scripts/ab_outputs.py --compare $out/ab_outputs_old.json $out/ab_outputs_new.json | tee -a $out/ab_outputs.log
