#!/bin/bash
# usage: gpu_quick.sh "<integrator> <flags>" ...   (env SPP, WORKLOAD, NOTEST, OUT: directory for the JSON lines and stderr)
OUT=${OUT:-$(mktemp -d)}
mkdir -p "$OUT"
[ -z "$NOTEST" ] && python -m pytest tests -m gpu -q -x 2>&1 | tail -4
for cfg in "$@"; do set -- $cfg
python bench.py --workload ${WORKLOAD:-c3} --spp ${SPP:-8} --steps 3 --warmup 2 --no-cpu-baseline --integrator $1 --flags $2 2>"$OUT/err.log" | tee "$OUT/bench_${WORKLOAD:-c3}_i$1_f$2.json" | python -c "
import json,sys
for l in sys.stdin:
    d=json.loads(l); r=d['roofline']
    print('${WORKLOAD:-c3} ${SPP:-8}spp integrator $1 flags $2: %.1f Mrays/s  %.2f ms/step  kernel %.2f ms  frac %.3f  e2e %.1f  spp/s %.1f M rays/frame %d launches %d' % (d['value'], d['ms_per_step'], r.get('kernel_ms', r.get('frame', {}).get('kernel_ms', 0)), r['frac'], d['e2e']['value'], d['spp_per_s']/1e6, d['rays_per_frame'], d['gpu_launches']))
"
tail -3 "$OUT/err.log"
done
echo "results in $OUT"
