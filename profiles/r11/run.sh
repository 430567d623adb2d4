#!/bin/bash
# Round 11: one carry kernel for the time-sharded passes and one packing path for the block phases, against the parent
# commit's library, in one session on one GPU:
#   profiles/r11/run.sh <parent libmoihgp.so> <output directory>
# 1. profiles/r11/ab_outputs.py under both libraries, compared byte for byte;
# 2. bench.py on c3, c4 and c5 alternating the parent library and this one (old, new, new, old) with --dump-outputs,
#    the dumps hashed (the arrays themselves are deleted);
# 3. the GPU test suite and smoke().
old=$(realpath $1); out=$2
mkdir -p $out
tmp=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv,noheader | head -1 | tee $out/card.txt
MOIHGP_B200_LIB=$old python profiles/r11/ab_outputs.py run $tmp/ab_old > $out/ab_outputs.log 2>&1
python profiles/r11/ab_outputs.py run $tmp/ab_new >> $out/ab_outputs.log 2>&1
python profiles/r11/ab_outputs.py compare $tmp/ab_old $tmp/ab_new | tee -a $out/ab_outputs.log
rm -rf $tmp/ab_old $tmp/ab_new
for wl in c3 c4 c5; do
  run=0
  for b in old new new old; do
    run=$((run + 1))
    lib=""; [ $b = old ] && lib=$old
    MOIHGP_B200_LIB=$lib python bench.py --gpus 1 --workload $wl --no-cpu --no-also --no-e2e --dump-outputs $tmp/dump_${wl}_${run}_$b \
      > $out/bench_${wl}_${run}_$b.json 2> $out/bench_${wl}_${run}_$b.err
  done
done
python - $out $tmp <<'PY' | tee $out/summary.txt
import glob, hashlib, json, os, sys
out, tmp = sys.argv[1], sys.argv[2]
print("card, power limit, max SM clock, driver:", open(os.path.join(out, "card.txt")).read().strip())
print("wl   run  build  ms_per_step  launches  dumps")
for f in sorted(glob.glob(os.path.join(out, "bench_c*.json"))):
    wl, run, b = os.path.basename(f)[6:-5].split("_")
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except (IndexError, ValueError):
        print("%-4s %-4s %-6s failed: %s" % (wl, run, b, open(f[:-5] + ".err").read().strip().splitlines()[-1:]))
        continue
    files = sorted(glob.glob(os.path.join(tmp, "dump_%s_%s_%s" % (wl, run, b), "*.npy")))
    h = hashlib.sha256(b"".join(hashlib.sha256(open(p, "rb").read()).digest() for p in files)).hexdigest()[:16]
    print("%-4s %-4s %-6s %11.4f  %8s  %s (%d files)" % (wl, run, b, d["ms_per_step"], d.get("gpu_launches"), h, len(files)))
PY
rm -rf $tmp
python -m pytest -m gpu tests -q -p no:cacheprovider > $out/gpu_tests.log 2>&1
tail -1 $out/gpu_tests.log
python -m pytest -m gpu tests/test_gpu_block_carry.py -v -p no:cacheprovider > $out/new_tests.log 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > $out/smoke.log 2>&1
tail -1 $out/smoke.log
