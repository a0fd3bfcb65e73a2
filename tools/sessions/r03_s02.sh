#!/bin/bash
# r03 session 2: interleaved A/B of the previous build against this tree (K1 ring 120 KB at n <= 10, K2 ring 100 KB at
# n <= 10), an A-vs-A of the previous build, then bench.py alternating the two builds with the outputs compared bit for bit
OUT=${1:?usage: $0 OUTPUT_DIR}
export OUT
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03_card_s02.txt
L=beyond_deep_ensembles_b200/lib
S=10x100000000,5x200000000,8x100000000,12x80000000
timeout 150 python tools/ab_libs.py --a $L/prev/libbde_b200.so --b $L/new/libbde_b200.so --shapes $S,4x250000000,6x160000000,7x140000000,9x110000000,11x90000000 --rounds 5 > $OUT/r03_ab_new.jsonl 2> $OUT/r03_ab_s02.err
echo "A=prev B=new rc=$?"; cat $OUT/r03_ab_new.jsonl
timeout 90 python tools/ab_libs.py --a $L/prev/libbde_b200.so --b $L/prev2/libbde_b200.so --shapes $S --rounds 5 > $OUT/r03_ab_aa.jsonl 2>> $OUT/r03_ab_s02.err
echo "A=prev B=prev2 rc=$?"; cat $OUT/r03_ab_aa.jsonl
tail -3 $OUT/r03_ab_s02.err
for i in 1 2 3; do
  for which in prev new; do
    extra=""; [ $i = 1 ] && extra="--dump-outputs $OUT/dump_$which"
    if [ $which = prev ]; then export BDE_B200_LIB=$PWD/$L/prev/libbde_b200.so; else unset BDE_B200_LIB; fi
    timeout 60 python bench.py --gpus 1 --steps 20 --warmup 3 --skip-extras $extra > $OUT/r03_bench_${which}_$i.json 2> $OUT/r03_bench_${which}_$i.err
    echo "bench $which $i rc=$?"; head -c 300 $OUT/r03_bench_${which}_$i.json; echo
  done
done
unset BDE_B200_LIB
python - <<'PY'
import glob, json, os, statistics, numpy as np
OUT = os.environ["OUT"]
names = sorted(os.path.basename(p) for p in glob.glob(f"{OUT}/dump_prev/*.npy"))
same = {n: bool(np.array_equal(np.load(f"{OUT}/dump_prev/{n}"), np.load(f"{OUT}/dump_new/{n}"))) for n in names}
print("bit-identical:", same, all(same.values()) and len(names) > 0)
for w in ("prev", "new"):
    recs = [json.loads(open(f"{OUT}/r03_bench_{w}_{i}.json").read().strip().splitlines()[-1]) for i in (1, 2, 3)]
    ms = [r["ms_per_step"] for r in recs]
    print(w, "ms_per_step", [round(m, 4) for m in ms], "median", round(statistics.median(ms), 4), "spread", round((max(ms) - min(ms)) / statistics.median(ms), 4),
          "kernels", {k: round(v["ms"], 4) for k, v in recs[0]["kernels"].items()})
PY
