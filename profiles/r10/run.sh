#!/bin/bash
# Round 10: time-sharded posterior sampling on one GPU, and the unchanged paths against the parent commit, in one session:
#   profiles/r10/run.sh <parent tree, built> <output directory>
# 1. scripts/ab_sample_outputs.py with both libraries (whole-sequence sampler, both variants, config-3 and config-4 shapes),
#    checksums compared; scripts/ab_outputs.py in both trees;
# 2. bench.py on c3 (the default line) and c4, alternating the parent tree and this one (old, new, new, old);
# 3. scripts/bench_time_shard_sample.py with one rank (the whole-sequence call, T = 8e6, S = 4);
# 4. the GPU test suite.
old=$1; out=$2
mkdir -p $out
here=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv,noheader | head -1 | tee $out/card.txt
cp scripts/ab_sample_outputs.py $old/scripts/
(cd $old && python scripts/ab_sample_outputs.py $here/$out/ab_sample_old.json) > $out/ab_sample.log 2>&1
python scripts/ab_sample_outputs.py $out/ab_sample_new.json >> $out/ab_sample.log 2>&1
python scripts/ab_outputs.py --compare $out/ab_sample_old.json $out/ab_sample_new.json | tee -a $out/ab_sample.log
(cd $old && python scripts/ab_outputs.py $here/$out/ab_outputs_old.json) > $out/ab_outputs.log 2>&1
python scripts/ab_outputs.py $out/ab_outputs_new.json >> $out/ab_outputs.log 2>&1
python scripts/ab_outputs.py --compare $out/ab_outputs_old.json $out/ab_outputs_new.json | tee -a $out/ab_outputs.log
for wl in c3 c4; do
  run=0
  for b in old new new old; do
    run=$((run + 1))
    if [ $b = old ]; then cd $old; else cd $here; fi
    python bench.py --gpus 1 --workload $wl --no-cpu --no-also --no-e2e > $here/$out/bench_${wl}_${run}_$b.json 2> $here/$out/bench_${wl}_${run}_$b.err
    cd $here
  done
done
python scripts/bench_time_shard_sample.py > $out/time_shard_sample_1gpu.jsonl 2> $out/time_shard_sample_1gpu.err
python -m pytest -m gpu tests -q -s -p no:cacheprovider > $out/gpu_tests.log 2>&1
tail -1 $out/gpu_tests.log
