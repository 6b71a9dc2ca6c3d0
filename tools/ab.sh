#!/bin/bash
# developer tool: A/B the variant builds of libsab200 on one box (device-resident bench)
#   AB_VARIANTS="_i16 _x"  suffixes of suffix_array_b200/libsab200<suffix>.so (built with `make variant`)
#   AB_MIB=256  AB_WORKLOAD=c2
for v in "" ${AB_VARIANTS}; do
  lib=suffix_array_b200/libsab200$v.so
  [ -f $lib ] || continue
  echo -n "variant '$v': "
  SAB200_LIB=$PWD/$lib python bench.py --workload ${AB_WORKLOAD:-c2} --n-mib ${AB_MIB:-256} --steps 2 --warmup 2 --no-search --no-cpu-baseline 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print(d['value'],'MB/s', d['ms_per_step'],'ms', 'pass GB/s',d['roofline']['achieved'], d['breakdown_ms'], d['config']['radix_passes'])"
done
