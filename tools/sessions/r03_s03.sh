#!/bin/bash
# r03 session 3: the whole GPU suite and smoke() on the final tree
OUT=${1:?usage: $0 OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03_card_s03.txt
timeout 480 python -m pytest tests -q -m gpu 2>&1 | tail -15 > $OUT/r03_pytest_gpu_n1.txt; echo "pytest rc=${PIPESTATUS[0]}"
cat $OUT/r03_pytest_gpu_n1.txt
timeout 90 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3 | tee $OUT/r03_smoke.txt
