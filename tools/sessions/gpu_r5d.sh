#!/bin/bash
# GPU session r5d: the Groth16 one-call prover after the assembly rework -- its tests, the tests that go through
# create_proof, and tools/groth16_prove_bench.py (four paths, per-kernel assembly times).
OUT=${1:?usage: gpu_r5d.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/gpu_r5d.txt 2>&1
timeout 300 python -m pytest -m gpu -q --maxfail=20 -p no:cacheprovider tests/test_gpu_groth16_prove.py tests/test_groth16_proof.py \
    tests/test_groth16_verify.py "tests/test_gpu_multidev.py::test_groth16_create_proof_places_g2_remotely" \
    "tests/test_gpu_fixed_base.py::test_groth16_setup_fixed_base_end_to_end" > "$OUT"/pytest_groth16_prove_r5d.log 2>&1
echo "pytest rc=$?"; tail -2 "$OUT"/pytest_groth16_prove_r5d.log; grep -E "^(FAILED|ERROR)" "$OUT"/pytest_groth16_prove_r5d.log | head
timeout 420 python tools/groth16_prove_bench.py --out "$OUT"/groth16_prove_r5d.jsonl > "$OUT"/groth16_prove_r5d.log 2>&1
echo "prove bench rc=$?"; grep -v -i warn "$OUT"/groth16_prove_r5d.log | tail -30 | cut -c1-260
