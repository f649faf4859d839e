#!/bin/bash
# same-box A/B of several builds of the library: tools/ab_libs.sh a.so b.so ...  (scan launch times per workload;
# WL="c3 c4", REPS="1 2", CHECK=1 also runs the tensor-core parity tests against each build)
keep=$(mktemp)
cp better-binary-quantization_b200/libbbq_b200.so "$keep"
for rep in ${REPS:-1 2}; do for lib in "$@"; do
  [ "$lib" -ef better-binary-quantization_b200/libbbq_b200.so ] || cp "$lib" better-binary-quantization_b200/libbbq_b200.so
  if [ "${CHECK:-0}" = 1 ] && [ "$rep" = 1 ]; then
    echo -n "$(basename $lib) parity: "
    timeout -s KILL 600 python -m pytest tests/test_gpu_parity.py tests/test_gpu_round2.py -x -q -k "mma or 4096 or large_k" 2>&1 | tail -1
  fi
  for w in ${WL:-c3 c4}; do
    echo -n "$(basename $lib) $w: "
    timeout -s KILL ${TMO:-300} python bench.py --workload $w --datagen device --no-cpu --no-secondary --steps ${STEPS:-5} ${EXTRA:-} 2>/dev/null | tail -1 | \
      python -c "import sys,json; d=json.loads(sys.stdin.read()); r=d['roofline']; print('QPS', round(d['value']), 'ms/step', round(d['ms_per_step'],3), 'e2e ms/step', round(d['e2e']['ms_per_step'],4), 'scan launch ms', round(r['avg_scan_launch_ms'],4), 'passes', r.get('passes_over_shard'), 'frac', round(r['frac'],3))"
  done
done; done
cp "$keep" better-binary-quantization_b200/libbbq_b200.so
