#!/bin/bash
# GPU session r4c: the fixed-base library as committed -- whole GPU suite, the fixed-base sweep (device leg timed on a
# stream of its own), smoke, the default bench line.
OUT=${1:?usage: gpu_r4c.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/gpu_r4c.txt 2>&1
timeout 1500 python -m pytest tests -m gpu -q --maxfail=30 -p no:cacheprovider > "$OUT"/pytest_gpu_r4c.log 2>&1
echo "pytest rc=$?"; tail -3 "$OUT"/pytest_gpu_r4c.log; grep -E "^(FAILED|ERROR)" "$OUT"/pytest_gpu_r4c.log | head -20
timeout 900 python tools/fixed_base_sweep.py --out "$OUT"/sweep_fixed_base_r4c.jsonl > "$OUT"/sweep_fixed_base_r4c.log 2>&1
echo "sweep rc=$?"; tail -3 "$OUT"/sweep_fixed_base_r4c.log | cut -c1-300
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/smoke_r4c.log 2>&1; echo "smoke rc=$?"; tail -1 "$OUT"/smoke_r4c.log
timeout 400 python bench.py --gpus 1 > "$OUT"/bench_r4c.json 2> "$OUT"/bench_r4c.err
echo "bench rc=$?"; tail -c 600 "$OUT"/bench_r4c.json; tail -2 "$OUT"/bench_r4c.err
