#!/bin/bash
# GPU session r5e: the whole GPU suite, smoke and the default bench line on the final library.
OUT=${1:?usage: gpu_r5e.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/gpu_r5e.txt 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/smoke_r5e.log 2>&1; echo "smoke rc=$?"; tail -1 "$OUT"/smoke_r5e.log
timeout 200 python bench.py --gpus 1 > "$OUT"/bench_r5e_n1.json 2> "$OUT"/bench_r5e.err
echo "bench rc=$?"; head -c 300 "$OUT"/bench_r5e_n1.json; echo; tail -2 "$OUT"/bench_r5e.err
timeout 420 python -m pytest tests -m gpu -q --maxfail=30 -p no:cacheprovider > "$OUT"/pytest_gpu_r5e.log 2>&1
echo "pytest rc=$?"; tail -2 "$OUT"/pytest_gpu_r5e.log; grep -E "^(FAILED|ERROR)" "$OUT"/pytest_gpu_r5e.log | head -20
