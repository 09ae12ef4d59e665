# K1 trace-writer ceiling: the default GlobalMCMC workload (65,536 chains x 1e4 iterations) with a chain-major trace,
# a time-major trace and no trace, alternated three times.  chain - none is the most any change to the chain-major
# writer can win.  LIB selects the library (default: the in-tree build).
LIB=${LIB:-$PWD/gl-abc-mcmc_b200/csrc/libglabc.so}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
for rep in 1 2 3; do
  for layout in chain time none; do
    GLABC_LIB=$LIB python bench.py --layout $layout --no-cpu --no-e2e --no-extra --no-other-configs --no-ref-python 2>/dev/null |
      python -c "import json,sys; d=json.loads(sys.stdin.read()); print('$layout', d['value'], d['roofline']['kernel_ms'])"
  done
done
