#!/bin/bash
# A/B: suffix-sorting of query batches on/off on the headline workload
summ='import json,sys
d=json.loads(sys.stdin.readlines()[-1]); l=d.get("locate") or {}
print("value %.1fM q/s  %.2f ms | e2e %.1fM q/s %.2f ms | frac %.3f | locate e2e %.1fM q/s %.2f ms (walk kernels %.2f ms)" % (d["value"]/1e6, d["ms_per_step"], d["e2e"]["value"]/1e6, d["e2e"]["ms_per_step"], d["roofline"]["frac"], l.get("value",0)/1e6, l.get("ms_per_step",0), l.get("kernel_ms_locate",0)))'
for sort in 0 1; do
  echo "== GDX_SORT_QUERIES=$sort"
  GDX_SORT_QUERIES=$sort python bench.py --steps 5 --warmup 3 --no-cpu-baseline | python -c "$summ"
done
