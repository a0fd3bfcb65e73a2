#!/bin/bash
# r03 session 1: streaming ceilings at n = 10 (tools/microbench/stream_mix.cu), then interleaved A/B of K1 ring
# candidates (lane-per-row producer, 80 KB / 120 KB ring) and of K2 ring depths against the previous build
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03_card.txt
timeout 120 tools/microbench/stream_mix 9 > $OUT/r03_stream_mix.jsonl 2> $OUT/r03_stream_mix.err; echo "stream_mix rc=$?"
cat $OUT/r03_stream_mix.jsonl
L=beyond_deep_ensembles_b200/lib
S=10x100000000,5x200000000,8x100000000,12x80000000
for b in prev2 v80 v120; do
  timeout 300 python tools/ab_libs.py --a $L/prev/libbde_b200.so --b $L/$b/libbde_b200.so --shapes $S --rounds 5 > $OUT/r03_ab_k1_$b.jsonl 2>> $OUT/r03_ab.err
  echo "k1 A=prev B=$b rc=$?"; cat $OUT/r03_ab_k1_$b.jsonl
done
for r in 80 100 160; do
  timeout 300 python tools/ab_libs.py --a $L/prev/libbde_b200.so --b $L/prev2/libbde_b200.so --tune-b ring_kb=$r --shapes $S --rounds 5 > $OUT/r03_ab_ring_$r.jsonl 2>> $OUT/r03_ab.err
  echo "k2 ring_kb=$r rc=$?"; cat $OUT/r03_ab_ring_$r.jsonl
done
tail -5 $OUT/r03_ab.err
