#!/bin/bash
# Developer aid: A/B several builds of libodhead in ONE GPU session, since box-to-box variance is ~8 %. Each build is an
# objectdetection_b200/libodhead_<name>.so, e.g. the library of another commit or a build.build_variant build.
# Usage: bash tools/ab_libs.sh name1 name2 ...   ("base" = libodhead.so)
for rep in 1 2; do
for name in "$@"; do
  lib=$PWD/objectdetection_b200/libodhead_$name.so
  [ "$name" = base ] && lib=$PWD/objectdetection_b200/libodhead.so
  ODHEAD_LIB=$lib python bench.py --steps 100 --warmup 5 --no-cpu-baseline 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1])
s=d['roialign_standalone']
print('%-8s'%'$name', 'step_ms %.4f'%d['ms_per_step'], 'p14pipe %.4f (%.3f)'%(d['roofline']['ms_per_launch'], d['roofline']['frac']), 'sa_p7 %.4f (%.3f) sa_p14 %.4f (%.3f)'%(s['p7']['ms'],s['p7']['frac'],s['p14']['ms'],s['p14']['frac']))"
done
done
