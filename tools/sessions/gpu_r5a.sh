#!/bin/bash
# GPU session r5a: the Groth16 one-call prover -- its own tests and the existing tests that go through create_proof.
OUT=${1:?usage: gpu_r5a.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT"/gpu_r5a.txt 2>&1
timeout 1200 python -m pytest -m gpu -q --maxfail=20 -p no:cacheprovider tests/test_gpu_groth16_prove.py tests/test_groth16_proof.py \
    tests/test_groth16_verify.py "tests/test_gpu_multidev.py::test_groth16_create_proof_places_g2_remotely" \
    "tests/test_gpu_fixed_base.py::test_groth16_setup_fixed_base_end_to_end" > "$OUT"/pytest_r5a.log 2>&1
echo "pytest rc=$?"; tail -3 "$OUT"/pytest_r5a.log; grep -E "^(FAILED|ERROR)|Error|assert" "$OUT"/pytest_r5a.log | head -30
