#!/bin/bash
# Round-2 A/B call: tests, then same-box comparisons —
#   C2 headline: round-1 library (lib_base) vs current;  C3/C5: one vs two paths per lane (RT_PATHS_PER_LANE).
set -u
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?"; tail -5 gpurun_out/pytest_gpu.log
line() { python -c "
import json,sys
for l in sys.stdin:
    d=json.loads(l); r=d['roofline']; e=d.get('e2e') or {}
    print('$1', d['config']['workload'][:3], d['config']['kernel'][:5], 'ms/step %.3f' % d['ms_per_step'], 'Mrays/s %.1f' % d['value'], 'e2e_ms %.3f' % e.get('ms_per_frame',0), 'frac %.4f' % r['frac'])
"; }
B="--no-extras --no-cpu-baseline"
for rep in 1 2; do
  RT_LIB_VARIANT=base python bench.py --workload c2 --steps 40 $B --no-e2e 2>>gpurun_out/bench.err | line "base  "
  python bench.py --workload c2 --steps 40 $B --no-e2e 2>>gpurun_out/bench.err | line "new   "
done
for np in 1 2; do
  for fm in "" "--fast-math"; do
    RT_PATHS_PER_LANE=$np python bench.py --workload c3 --steps 3 $B --no-e2e $fm 2>>gpurun_out/bench.err | line "np=$np"
    RT_PATHS_PER_LANE=$np python bench.py --workload c5 --steps 3 $B --no-e2e $fm 2>>gpurun_out/bench.err | line "np=$np"
  done
done
tail -5 gpurun_out/bench.err
