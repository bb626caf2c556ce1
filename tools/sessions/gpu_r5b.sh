#!/bin/bash
# GPU session r5b: the Groth16 one-call prover -- whole GPU suite, the prover benchmark (three paths alternating),
# smoke, the default bench line.
OUT=${1:?usage: gpu_r5b.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/gpu_r5b.txt 2>&1
timeout 400 python bench.py --gpus 1 > "$OUT"/bench_r5b_n1.json 2> "$OUT"/bench_r5b.err
echo "bench rc=$?"; tail -c 700 "$OUT"/bench_r5b_n1.json; tail -2 "$OUT"/bench_r5b.err
timeout 900 python tools/groth16_prove_bench.py --out "$OUT"/groth16_prove_r5b.jsonl > "$OUT"/groth16_prove_r5b.log 2>&1
echo "prove bench rc=$?"; tail -30 "$OUT"/groth16_prove_r5b.log | cut -c1-400
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/smoke_r5b.log 2>&1; echo "smoke rc=$?"; tail -1 "$OUT"/smoke_r5b.log
timeout 1500 python -m pytest tests -m gpu -q --maxfail=30 -p no:cacheprovider > "$OUT"/pytest_gpu_r5b.log 2>&1
echo "pytest rc=$?"; tail -3 "$OUT"/pytest_gpu_r5b.log; grep -E "^(FAILED|ERROR)" "$OUT"/pytest_gpu_r5b.log | head -20
