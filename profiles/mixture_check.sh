#!/bin/bash
# Validation of the Gaussian-mixture plugin on one B200: build, smoke, the whole GPU suite, the default bench line and
# its --dump-outputs of this build and (with PARENT_LIB=<libkissmcmc_cuda.so of the parent commit>) of the parent,
# compared file for file, then profiles/mixture_bench.py.
# Usage: profiles/mixture_check.sh OUTDIR      (logs, bench lines and the mixture_bench JSON go to OUTDIR)
OUT=${1:?usage: profiles/mixture_check.sh OUTDIR}
mkdir -p "$OUT"
DUMPS=$(mktemp -d)    # the dumped outputs are large: compared here, not kept
trap 'rm -rf "$DUMPS"' EXIT
python -c 'import __graft_entry__ as g; g.build()' > $OUT/mixture_build.log 2>&1 || { tail -20 $OUT/mixture_build.log; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv,noheader | tee $OUT/mixture_gpu.txt
timeout 120 python __graft_entry__.py smoke > $OUT/mixture_smoke.log 2>&1; tail -1 $OUT/mixture_smoke.log
timeout 900 python -m pytest tests -m gpu -q -rs --durations=12 > $OUT/mixture_pytest_gpu.log 2>&1
echo "pytest exit $?" >> $OUT/mixture_pytest_gpu.log
tail -16 $OUT/mixture_pytest_gpu.log
for arm in new parent; do
  if [ "$arm" = parent ]; then [ -n "$PARENT_LIB" ] || continue; export KMC_LIB=$PARENT_LIB; fi
  timeout 300 python bench.py --gpus 1 --steps 3 --warmup 1 --dump-outputs $DUMPS/dump_$arm \
    > $OUT/bench_$arm.json 2> $OUT/bench_$arm.err
  echo "bench $arm exit $?"; tail -1 $OUT/bench_$arm.json | cut -c1-300
  unset KMC_LIB
done
if [ -n "$PARENT_LIB" ]; then
  DUMPS=$DUMPS python - <<'PY' | tee $OUT/mixture_dump_compare.txt
import numpy as np, pathlib
import os
d = pathlib.Path(os.environ["DUMPS"])
a, b = d / "dump_new", d / "dump_parent"
names = sorted(p.name for p in a.glob("*.npy"))
same = [np.array_equal(np.load(a / n), np.load(b / n), equal_nan=True) for n in names]
print("dump-outputs vs parent:", dict(zip(names, same)), "IDENTICAL" if names and all(same) else "DIFFERENT")
PY
fi
timeout 900 python profiles/mixture_bench.py > $OUT/mixture_bench.json 2> $OUT/mixture_bench.err
echo "mixture_bench exit $?"; tail -3 $OUT/mixture_bench.err; cut -c1-400 $OUT/mixture_bench.json
