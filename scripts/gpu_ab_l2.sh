# L2-reuse A/B of step-library builds on one box: VARIANTS="BASE NEW" bash scripts/gpu_ab_l2.sh
# (libs in build_ab/lib<v>.so).  Runs scripts/l2_reuse_probe.py for every build, then the headline
# bench line REPS times per build, alternating builds.  BENCH_ARGS="" gives bench.py's default run.
# Results go to $OUT (default build_ab/out).
OUT=${OUT:-build_ab/out}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv,noheader | tee "$OUT/card.txt"
if [ "${PROBE:-1}" = "1" ]; then
  for v in ${VARIANTS:-BASE NEW}; do
    MARLNAV_B200_LIB=$PWD/build_ab/lib$v.so timeout ${TMO:-300} python scripts/l2_reuse_probe.py --label $v --out "$OUT/l2_reuse_probe.jsonl" \
      | python -c "import json,sys; [print('PROBE', d['label'], d['shape'], d['us_per_step'], d['ns_per_env']) for d in map(json.loads, sys.stdin)]"
  done
fi
for rep in $(seq ${REPS:-3}); do for v in ${VARIANTS:-BASE NEW}; do
MARLNAV_B200_LIB=$PWD/build_ab/lib$v.so timeout ${TMO:-300} python bench.py ${BENCH_ARGS---no-cpu-baseline --no-ref-cuda --no-configs --no-strong --e2e-steps 3} 2>/dev/null | tee -a "$OUT/bench_$v.jsonl" \
  | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('AB $v us_per_step', round(d['ms_per_step']*1000,2), 'clocks', d.get('clocks'))" | tee -a "$OUT/ab.log"
done; done
