#!/bin/bash
# tools/ab.sh LIB... -- time the playout + greedy kernels with alternative builds of the library (on the GPU box:
# overwrites the in-tree .so of the scratch copy).  Per build: value, ms_per_step, a launch alone, the two e2e figures
# and the SM clocks sampled during the timed steps.
for lib in "$@"; do
  cp "$lib" subproc_b200/libothello_b200.so
  echo "== $lib"
  python bench.py --no-cpu-baseline --no-extra --steps 40 2>&1 | python -c "
import sys, json
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
print('playout', '%.4g' % d['value'], d['ms_per_step'], 'alone', d['roofline']['kernel_alone_ms'], 'e2e', '%.4g' % d['e2e']['value'],
      'e2e_std', '%.4g' % d['e2e']['standard_opening']['value'], 'clocks', json.dumps(d['clocks']))"
done
