# K1 tile loop A/B on one GPU: the parent library (PARENT, built from the previous commit) against the in-tree build,
# alternated, on the default GlobalMCMC workload (65,536 chains x 1e4 iterations) with a chain-major, a time-major and no
# trace, and on GLMCMC (K2 shares the trace writer).  Then both dump the outputs of the same seeded run for a byte compare.
#   PARENT=/path/to/libglabc.so [CASES="chain glmcmc ..."] bash profiles/micro/k1_tile_ab.sh OUTDIR
PARENT=${PARENT:?path of the parent build}
NEW=$PWD/gl-abc-mcmc_b200/csrc/libglabc.so
OUT=${1:?output directory}
FLAGS="--no-cpu --no-e2e --no-extra --no-other-configs --no-ref-python"
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
one() {  # variant library args...
  local v=$1 lib=$2; shift 2
  GLABC_LIB=$lib python bench.py $FLAGS "$@" 2>/dev/null | tee -a $OUT/ab_$v.jsonl |
    python -c "import json,sys; d=json.loads(sys.stdin.read()); print('$v', '$*', d['value'], d['roofline']['kernel_ms'])"
}
CASES=${CASES:-"chain chain chain time none glmcmc time none glmcmc"}
for c in $CASES; do
  case $c in chain|time|none) args="--layout $c" ;; *) args="--sampler $c" ;; esac
  one parent $PARENT $args
  one new $NEW $args
done
# parent2: a second parent run, to tell an order-dependent reduction (summary.npy: glabc_summarize adds its blocks'
# float64 partial sums with atomicAdd) from a change of results
for v in parent new parent2; do
  lib=$PARENT; [ $v = new ] && lib=$NEW
  GLABC_LIB=$lib python bench.py $FLAGS --steps 3 --warmup 1 --dump-outputs $OUT/dump_$v > /dev/null 2>&1
done
for f in trace theta y stats summary; do
  cmp $OUT/dump_parent/$f.npy $OUT/dump_new/$f.npy && echo "$f.npy byte-equal"
done
cmp $OUT/dump_parent/summary.npy $OUT/dump_parent2/summary.npy && echo "summary.npy parent run-to-run byte-equal"
