#!/bin/bash
# Mutation check of tests/test_gpu_parameter_box.py: each patch under profiles/r12/mutants/ breaks k_setup (setup.cu) in one
# way; the patched copy is built into a side library with scripts/build_variant.sh (outside the product library) and the
# new file and the rest of the GPU suite run against it through MOIHGP_B200_LIB.
#   profiles/r12/run_mutants.sh <output directory> [<mutant name> ...]   (default: every patch)
out=$1; shift
names="$*"
mkdir -p $out
tmp=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv,noheader | head -1 > $out/card.txt
[ -z "$names" ] && names=$(for p in profiles/r12/mutants/*.patch; do basename $p .patch; done)
for m in $names; do
  p=profiles/r12/mutants/$m.patch
  lib=$PWD/multioutputihgp_b200/lib/ab/libmoihgp_$m.so
  if [ ! -f $lib ]; then
    mkdir -p $tmp/$m
    patch -s -p1 -o $tmp/$m/setup.cu < $p
    scripts/build_variant.sh $m "-I$PWD/multioutputihgp_b200/csrc" $tmp/$m/setup.cu > /dev/null
  fi
  MOIHGP_B200_LIB=$lib python -m pytest tests/test_gpu_parameter_box.py -m gpu -q -p no:cacheprovider -rf 2>&1 | grep -E "^(FAILED|ERROR) |(passed|failed)" > $out/${m}_new_file.log
  MOIHGP_B200_LIB=$lib python -m pytest tests -m gpu -q -p no:cacheprovider -rf --ignore=tests/test_gpu_parameter_box.py 2>&1 | grep -E "^(FAILED|ERROR) |(passed|failed)" > $out/${m}_rest_of_suite.log
done
rm -rf $tmp
python - $out <<'PY' | tee $out/summary.txt
import collections, glob, os, re, sys
out = sys.argv[1]
print("card, power limit, max SM clock, driver:", open(os.path.join(out, "card.txt")).read().strip())
for f in sorted(glob.glob(os.path.join(out, "*_new_file.log"))):
    m = os.path.basename(f)[:-len("_new_file.log")]
    for part in ("new_file", "rest_of_suite"):
        text = open(os.path.join(out, "%s_%s.log" % (m, part))).read()
        last = text.strip().splitlines()[-1] if text.strip() else "(no output)"
        failed = re.findall(r"^FAILED (\S+?)(?:\[| |$)", text, re.M)
        by = collections.Counter(failed)
        print("%-28s %-14s %s" % (m, part, last))
        for t, n in sorted(by.items()):
            print("    %3d x %s" % (n, t))
PY
