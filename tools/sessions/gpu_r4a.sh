#!/bin/bash
# GPU session r4a: fixed-base batch scalar multiplication -- whole GPU suite (with tests/test_gpu_fixed_base.py), the
# fixed-base sweep, smoke, the default bench line.
OUT=${1:?usage: gpu_r4a.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/gpu_r4a.txt 2>&1
timeout 1500 python -m pytest tests -m gpu -q --maxfail=30 -p no:cacheprovider > "$OUT"/pytest_gpu_r4a.log 2>&1
echo "pytest rc=$?"; tail -3 "$OUT"/pytest_gpu_r4a.log; grep -E "^(FAILED|ERROR)" "$OUT"/pytest_gpu_r4a.log | head -20
timeout 900 python tools/fixed_base_sweep.py --out "$OUT"/sweep_fixed_base_r4a.jsonl > "$OUT"/sweep_fixed_base_r4a.log 2>&1
echo "sweep rc=$?"; tail -3 "$OUT"/sweep_fixed_base_r4a.log | cut -c1-300
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/smoke_r4a.log 2>&1; echo "smoke rc=$?"; tail -1 "$OUT"/smoke_r4a.log
timeout 400 python bench.py --gpus 1 > "$OUT"/bench_r4a.json 2> "$OUT"/bench_r4a.err
echo "bench rc=$?"; tail -c 600 "$OUT"/bench_r4a.json; tail -2 "$OUT"/bench_r4a.err
