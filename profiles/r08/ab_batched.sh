#!/bin/bash
# A/B of multioutputihgp_b200/batched.py against another version of the file (here: the parent commit's), on one GPU:
# the GPU suite under each version, then bench.py on c3, c4 and c5, alternating old, new, new, old, old, new, with
# --dump-outputs.  Restores the new file at the end; prints the summary and deletes the dumps after hashing them.
#   profiles/r08/ab_batched.sh <old batched.py> <output directory>
old=$1; out=$2
mkdir -p $out
new=$out/batched_new.py
cp multioutputihgp_b200/batched.py $new
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv,noheader | head -1 > $out/card.txt
use() { cp $1 multioutputihgp_b200/batched.py; }

use $old
python -m pytest -m gpu -q -p no:cacheprovider --ignore=tests/test_sequences_arguments.py > $out/gpu_tests_old.log 2>&1
use $new
python -m pytest -m gpu -q -p no:cacheprovider > $out/gpu_tests_new.log 2>&1

for wl in c3 c4 c5; do
  run=0
  for b in old new new old old new; do
    run=$((run + 1))
    if [ $b = old ]; then use $old; else use $new; fi
    python bench.py --gpus 1 --workload $wl --no-cpu --no-also --no-e2e --dump-outputs $out/dump_${wl}_${run}_$b \
      > $out/bench_${wl}_${run}_$b.json 2> $out/bench_${wl}_${run}_$b.err
  done
done
use $new

python - $out <<'PY' | tee $out/summary.txt
import glob, hashlib, json, os, sys
out = sys.argv[1]
print("card, power limit, max SM clock, driver:", open(os.path.join(out, "card.txt")).read().strip())
for b in ("old", "new"):
    print("pytest -m gpu (%s):" % b, open(os.path.join(out, "gpu_tests_%s.log" % b)).read().strip().splitlines()[-1])
print("wl   run  build  ms_per_step  launches  dumps")
for f in sorted(glob.glob(os.path.join(out, "bench_c*.json"))):
    wl, run, b = os.path.basename(f)[6:-5].split("_")
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except (IndexError, ValueError):
        print("%-4s %-4s %-6s failed: %s" % (wl, run, b, open(f[:-5] + ".err").read().strip().splitlines()[-1:]))
        continue
    files = sorted(glob.glob(os.path.join(out, "dump_%s_%s_%s" % (wl, run, b), "*.npy")))
    h = hashlib.sha256(b"".join(hashlib.sha256(open(p, "rb").read()).digest() for p in files)).hexdigest()[:16]
    print("%-4s %-4s %-6s %11.4f  %8s  %s (%d files)" % (wl, run, b, d["ms_per_step"], d.get("gpu_launches"), h, len(files)))
PY
rm -rf $out/dump_*
