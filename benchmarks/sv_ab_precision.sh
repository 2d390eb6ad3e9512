# A/B of shared-variance scoring kernel builds with the float64 oracle check (bench.py config 4, no secondary / CPU legs).
#   bash benchmarks/sv_ab_precision.sh lib1.so default ...   (libraries under benchmarks/bin/; "default" = the in-tree build)
cd "$(dirname "$0")/.."
for lib in "$@"; do
  if [ "$lib" = "default" ]; then unset SSP_B200_LIB; else export SSP_B200_LIB=$(pwd)/benchmarks/bin/$lib; fi
  timeout 300 python bench.py --steps 3 --warmup 2 --no-cpu-baseline --no-secondary 2>&1 | tail -1 | python -c "import sys,json; l=json.loads(sys.stdin.read()); c=l['check']; print('$lib', 'kernel_ms', round(l['roofline']['kernel_ms'],1), 'sm_mhz', l['clocks']['sm_mhz'], 'W', l['clocks'].get('power_w_max'), 'rel', '%.3g' % c['oracle_max_rel'], 'llr', '%.3g' % c['oracle_max_llr_abs'], 'scoring_rel', '%.3g' % c['oracle_scoring_only_max_rel'])"
done
