#!/bin/bash
# r03 session 4: full bench.py lines (paths section included) of the previous build and of the final tree
OUT=${1:?usage: $0 OUTPUT_DIR}
export OUT
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03_card_s04.txt
L=beyond_deep_ensembles_b200/lib
for which in prev new; do
  if [ $which = prev ]; then export BDE_B200_LIB=$PWD/$L/prev/libbde_b200.so; else unset BDE_B200_LIB; fi
  timeout 270 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/r03_bench_full_$which.json 2> $OUT/r03_bench_full_$which.err
  echo "bench $which rc=$?"; head -c 400 $OUT/r03_bench_full_$which.json; echo
done
unset BDE_B200_LIB
python - <<'PY'
import json, os
OUT = os.environ["OUT"]
a, b = (json.loads(open(f"{OUT}/r03_bench_full_{w}.json").read().strip().splitlines()[-1]) for w in ("prev", "new"))
print("step", a["ms_per_step"], b["ms_per_step"])
def flat(d, p=""):
    for k, v in d.items():
        if isinstance(v, dict): yield from flat(v, p + k + ".")
        elif isinstance(v, (int, float)) and ("ms" in k): yield p + k, v
pa, pb = dict(flat(a.get("paths", {}))), dict(flat(b.get("paths", {})))
for k in sorted(pa):
    if k in pb and pa[k]: print(f"{k}: {pa[k]:.4f} -> {pb[k]:.4f} ({pb[k] / pa[k] - 1:+.2%})")
PY
