"""bench.py's output contract, checked on CPU through the reference arm (the only arm that runs without a GPU):
stdout carries exactly ONE JSON line with the keys its readers rely on; the CPU arm describes its bounded sample.
On the GPU: what --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    env = dict(os.environ, ZKM_BENCH_CPU_LOG_N="13")            # a 2^13-point sample keeps this test to seconds
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "ms" and j["higher_is_better"] is False
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in j, k
    assert "workload" in j["config"] and "2^24" in j["config"]["workload"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "2^13" in cb["sample"] and cb["value"] == j["value"]
    assert cb["runs"] == j["steps"] == 2 and j["warmup"] == 0 and cb["host_threads"] >= 1
    # the timed region the line claims (steps x ms_per_step of the sample actually run) fits the wall clock of the run
    assert sum(cb["run_ms"]) / 1e3 <= j["wall_s"]


def test_reference_arm_ignores_an_inherited_single_thread_openmp_setting():
    """torchrun exports OMP_NUM_THREADS=1 to its children; the CPU arm passes its thread count explicitly."""
    env = dict(os.environ, ZKM_BENCH_CPU_LOG_N="13", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    j = json.loads(r.stdout.strip().splitlines()[-1])
    assert j["cpu_baseline"]["host_threads"] == len(os.sched_getaffinity(0))
    assert j["e2e"] == {"value": j["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["vs_baseline"] is None                                # BASELINE.md publishes no number for this metric


def test_non_zero_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", ZKM_BENCH_CPU_LOG_N="13")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bench_rejects_arguments_it_cannot_honour(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra,
                           capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert r.returncode == 2 and r.stdout.strip() == "", (extra, r.stdout, r.stderr[-2000:])
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_repeat_exactly(tmp_path):
    """--dump-outputs: float64 files of exact u32 words, within 64 MB, equal to the CPU oracle on the bench's seeded
    inputs, and identical from one run to the next."""
    import numpy as np
    from oracle import capi
    log_n = 18
    env = dict(os.environ, ZKM_BENCH_LOG_N=str(log_n))
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                            "--skip-cpu", "--skip-proxy", "--skip-precompute", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-3000:]
        j = json.loads(r.stdout.strip().splitlines()[-1])
        assert j["steps"] == 2 and j["config"]["result_ok"] is True
        files = sorted(p.name for p in out.iterdir())
        assert files == ["msm_result_infinity.npy", "msm_result_xy.npy", "ntt_sample_index.npy", "ntt_sample_output.npy"]
        assert sum(p.stat().st_size for p in out.iterdir()) <= 64 << 20
        d = {f[:-4]: np.load(out / f) for f in files}
        for a in d.values():
            assert a.dtype == np.float64 and np.all(a == np.floor(a)) and a.min() >= 0 and a.max() < 2.0 ** 32
        dumps.append(d)
    a, b = dumps
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    words = lambda u64: u64.view(np.uint32).astype(np.float64)
    n = 1 << log_n
    want_xy, want_inf = capi.msm(0, 1, capi.progression(0, 1, 0x1234567, 0x89ABCDE, n),
                                 capi.random_scalars(0, n, seed=0x5EED0000 + log_n))
    assert np.array_equal(a["msm_result_xy"].ravel(), words(want_xy)) and a["msm_result_infinity"].tolist() == [float(want_inf)]
    rows = a["ntt_sample_index"].astype(np.int64)
    assert len(rows) == 1 << 16 and np.all(np.diff(rows) > 0) and rows[-1] < n
    want_ntt = capi.ntt(0, capi.random_field_elements(0, n, seed=0x5EED1000 + log_n))
    assert np.array_equal(a["ntt_sample_output"], words(np.ascontiguousarray(want_ntt[rows])))
