#!/bin/bash
# Usage: bash profiles/run_glue_ab.sh <output dir>
# A/B of the trace-kernel glue (shadow rays finished in the any-hit trace, single-rank bounce shaded from the partition output
# and the hit cache) against the previous library, on the default one-GPU workload.
#   base = pg2024-data-parallel-ray-tracing_b200/libdprt_base.so: `make` of the parent commit, copied beside libdprt.so
#   new  = the tree's libdprt.so
# Alternating runs of `bench.py --steps 20 --warmup 5 --skip-cpu`, image dumps of both (base twice: determinism with six samples
# in flight), then the summary. Results -> <output dir>/glue_*.
OUT=${1:?usage: bash profiles/run_glue_ab.sh <output dir>}; mkdir -p "$OUT"
BASE=pg2024-data-parallel-ray-tracing_b200/libdprt_base.so
NEW=pg2024-data-parallel-ray-tracing_b200/libdprt.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/glue_card.txt
for i in 1 2 3; do
  for v in base new; do
    lib=$BASE; [ $v = new ] && lib=$NEW
    dump=""; { [ $i -le 2 ] && [ $v = base ]; } || { [ $i -eq 1 ] && [ $v = new ]; } && dump="--dump-outputs $OUT/glue_dump_${v}_$i"
    DPRT_LIB=$lib timeout 300 python bench.py --steps 20 --warmup 5 --skip-cpu $dump > $OUT/glue_${v}_$i.json 2> $OUT/glue_${v}_$i.err
    echo "$v $i rc=$?"
  done
done
python - "$OUT" <<'PY'
import json, statistics as st, sys
import numpy as np
O = sys.argv[1]
print(open(f"{O}/glue_card.txt").read().strip())
vals = {"base": [], "new": []}
for v in ("base", "new"):
    for i in (1, 2, 3):
        try:
            d = json.loads(open(f"{O}/glue_{v}_{i}.json").read().strip().splitlines()[-1])
        except Exception as e:
            print(v, i, "no result", e); continue
        vals[v].append(d["value"])
        s = d["stages"]
        print(v, i, round(d["value"], 1), "Mrays/s", "gpu_launches", d["gpu_launches"], "cached/step", d["main_ray_queries_from_hit_cache_per_step"],
              {k: (round(s[k]["ms"] / d["steps"], 3), s[k]["launches"]) for k in s})
for v in vals:
    if vals[v]:
        print(v, "median", round(st.median(vals[v]), 1), "min", round(min(vals[v]), 1), "max", round(max(vals[v]), 1))
if vals["base"] and vals["new"]:
    print("median gain %.2f %%" % (100 * (st.median(vals["new"]) / st.median(vals["base"]) - 1)),
          "| slowest new beats fastest base:", min(vals["new"]) > max(vals["base"]))
def img(n):
    return np.load(f"{O}/glue_dump_{n}/image.npy").view(np.uint32)
try:
    print("image base_1 == base_2:", np.array_equal(img("base_1"), img("base_2")), "| base_1 == new_1:", np.array_equal(img("base_1"), img("new_1")))
except Exception as e:
    print("image compare failed", e)
PY
