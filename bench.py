#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BASELINE.json: "G1 MSM 2^24 ms; NTT 2^24 ms").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W

One step = one 2^24-point BLS12-381 G1 MSM (BASELINE.json configs[1]: the standalone G1 MSM
sweep; 2^24 is the size the metric is quoted on).  With N GPUs the 2^24 (base, scalar) pairs are
range-sharded N ways (strong scaling): every rank runs the full pipeline on its slice, the N
partial points are all-gathered over NCCL/NVLink and summed on every rank.  `value` is the device
time of a step with scalars and bases resident in HBM; `e2e` is the same step through the host
C-ABI call (`zkm_msm_registered`: scalars copied from pinned host memory, result read back; the
bases are the proving key, registered once -- /root/reference/benches/groth16.rs:107-115 reuses
`pk` across proofs).  The same run also reports the 2^24 Fr NTT (`ntt`), the stage breakdown of
the MSM, the roofline of the dominant kernel (bucket accumulation, integer pipe) and the CPU
baseline: the arkworks-0.3.0 algorithm restated in C++ (oracle/cpp), timed on this box's cores.

`--impl reference` times that CPU restatement (arkworks itself cannot be built: no Rust toolchain,
crates not vendored) with all host threads on a bounded sample and prints the same JSON line.

`--dump-outputs DIR` writes, after the run, what the last timed step returned (rank 0), as float64 .npy
files holding 32-bit words (exact) of arkworks' u64 limbs, so that two builds can be compared output for
output on the same seeded inputs:
  msm_result_xy.npy        (2, 2*L64) the affine MSM result x, y (Montgomery limbs as u32 words)
  msm_result_infinity.npy  (1,)       1.0 if the result is the point at infinity
  ntt_sample_index.npy     (S,)       sorted rows of the 2^LOG_N NTT output, a fixed seeded sample
  ntt_sample_output.npy    (S, 8)     those rows (Fr element, Montgomery, as u32 words)   [not with --skip-ntt]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = int(os.environ.get("ZKM_BENCH_LOG_N", "24"))
CURVE_NAME = os.environ.get("ZKM_BENCH_CURVE", "bls12_381")
CURVE_ID = {"bls12_381": 0, "bn254": 1}[CURVE_NAME]
L64 = {0: 6, 1: 4}[CURVE_ID]
MADS_PER_MODMUL = {0: 300, 1: 136}[CURVE_ID]      # 2 n^2 + n wide MADs, n = 12 / 8 32-bit limbs (SURVEY 8d)
ALGO_MODMULS_PER_POINT = 160                       # ceil(255/16) windows x 10 products (XYZZ mixed add), SURVEY 8d
METRIC = "G1 MSM 2^%d ms (%s)" % (LOG_N, "BLS12-381" if CURVE_ID == 0 else "BN254")
CPU_LOG_N = int(os.environ.get("ZKM_BENCH_CPU_LOG_N", str(LOG_N)))   # the CPU arm runs the REAL workload size by default


def int_pipe_peak():
    """Integer-pipe peak = the fastest measured issue rate of a 32x32->64 multiply-add on this pool's B200
    (tools/microbench/int_pipe_peak.cu, profiles/int_pipe_peak_r2.jsonl, SASS in profiles/int_pipe_peak_r2.sass.txt).
    Every wide form -- IMAD.WIDE.U32 with or without a 64-bit addend, the carry-chained IMAD.WIDE.U32.X, IMAD.HI --
    issues at ~31 per clock per SM; only the 32-bit IMAD (low half) reaches 61.  Round 1's 17 993 GMAD/s
    ("imad_wide", profiles/imad_peak_r1.jsonl) was an artefact: ptxas had hoisted the loop-invariant product, the loop
    measured IADD3 pairs (SASS in the same file)."""
    best, src = 0.0, None
    try:
        for line in open(os.path.join(ROOT, "profiles", "int_pipe_peak_r2.jsonl")):
            r = json.loads(line)
            if r.get("bench") in ("mul_wide", "imad_hi", "imad_wide_carry_chain") and r["Gops_s"] > best:
                best, src = r["Gops_s"], "%s @ %d warps/SM" % (r["sass"], r["warps_per_sm"])
    except Exception:
        pass
    if not best:
        best, src = 8994.4, "fallback: IMAD.WIDE.U32.X chain, profiles/int_pipe_peak_r2.jsonl as committed"
    return best, src


IMAD_PEAK_GMADS, IMAD_PEAK_SRC = int_pipe_peak()


def read_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads() -> int:
    """Threads the CPU arm uses: every core this process may run on (an inherited OMP_NUM_THREADS=1, as torchrun
    sets, is ignored: the thread count is passed to the oracle explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_baseline_run(runs: int, log_n: int):
    """The arkworks-0.3.0 MSM algorithm (C++ restatement, oracle/cpp) on the host cores, on the REAL workload size
    (2^24 points, ~15-35 s per run depending on the box), `runs` times; nothing is extrapolated."""
    import numpy as np
    from oracle import capi
    n = 1 << log_n
    threads = host_threads()
    bases = capi.progression(CURVE_ID, 1, 0x1234567, 0x89ABCDE, n)
    scal = capi.random_scalars(CURVE_ID, n, seed=0x5EED0000 + log_n)
    c_bits = capi.msm_window_bits(n)
    bits = 255 if CURVE_ID == 0 else 254
    windows = (bits + c_bits - 1) // c_bits      # window_starts = 0, c, 2c, ... < MODULUS_BITS
    times = []
    for _ in range(max(1, runs)):
        t0 = time.perf_counter()
        capi.msm(CURVE_ID, 1, bases, scal, threads=threads)
        times.append((time.perf_counter() - t0) * 1e3)
    ms = sum(times) / len(times)
    out = {
        "value": ms, "unit": "ms", "cores": int(min(threads, windows)), "kind": "port", "runs": len(times),
        "sample": "the full 2^%d-point MSM, %d run(s), %d threads requested explicitly (arkworks runs one task per window: "
                  "%d windows at c=%d, so at most %d threads work); arkworks-0.3.0 algorithm restated in C++ (oracle/cpp), "
                  "not the Rust binary" % (log_n, len(times), threads, windows, c_bits, windows),
        "host_threads": threads, "run_ms": times,
    }
    if log_n != LOG_N:
        out["value"] = ms * (1 << LOG_N) / n
        out["sample"] += "; ZKM_BENCH_CPU_LOG_N override: value scaled linearly from 2^%d" % log_n
    return out


def cpu_ntt_baseline(log_n: int):
    """ark-poly's in_order_fft_in_place restated (oracle/cpp), all host threads, the real 2^log_n transform."""
    from oracle import capi
    threads = host_threads()
    x = capi.random_field_elements(CURVE_ID, 1 << log_n, seed=0x5EED1000 + log_n)
    capi.ntt(CURVE_ID, x[: 1 << 16], threads=threads)          # warm the thread pool
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        capi.ntt(CURVE_ID, x, threads=threads)
        times.append((time.perf_counter() - t0) * 1e3)
    return {"value": min(times), "unit": "ms", "cores": threads, "kind": "port", "runs": len(times),
            "sample": "the full 2^%d transform, best of %d, %d threads" % (log_n, len(times), threads)}


def run_reference(args):
    """--impl reference: the CPU arm alone.  One REAL 2^24 MSM per step; the requested step / warm-up counts are upper
    bounds (a step costs ~15-35 s of all host cores): at most 2 timed steps and no warm-up, reported as run."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps = max(1, min(args.steps, 2 if CPU_LOG_N >= 23 else 5))
    t0 = time.perf_counter()
    base = cpu_baseline_run(steps, CPU_LOG_N)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": "ms", "n_gpus": args.gpus,
        "steps": steps, "warmup": 0, "requested_steps": args.steps, "requested_warmup": args.warmup,
        "ms_per_step": base["value"], "higher_is_better": False,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64-limb Montgomery integers (CPU)", "data": "synthetic",
        "config": {"workload": "G1 MSM, %s, 2^%d points, uniform scalars; CPU: arkworks-0.3.0 algorithm restated in C++ "
                               "(oracle/cpp), not the Rust binary" % (CURVE_NAME, LOG_N),
                   "note": "steps / warmup are what actually ran: every step is the full 2^%d MSM on all host cores"
                           % CPU_LOG_N},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": None,
    }
    line["wall_s"] = time.perf_counter() - t0
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--skip-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--skip-ntt", action="store_true")
    ap.add_argument("--skip-proxy", action="store_true", help="skip the Groth16 proof proxy leg")
    ap.add_argument("--skip-precompute", action="store_true", help="skip the precomputed-bases MSM leg")
    ap.add_argument("--skip-single-process", action="store_true", help="skip the one-process-N-GPUs leg (N > 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: this benchmark has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # host-side barrier for the one-process-N-GPUs leg: an NCCL barrier would keep a spinning kernel on every waiting GPU
        cpu_group = dist.new_group(backend="gloo")

    import zkmember_b200 as zkm
    from zkmember_b200 import _lib
    zkm.init(local_rank)
    L = _lib.lib()
    # a dedicated (non-default) stream: the library launches on exactly this stream, so the
    # torch.cuda.Event pairs below bracket its kernels (handle 0 would mean "library's own stream")
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    sp = ctypes.c_void_p(stream)

    n_total = 1 << LOG_N
    n_local = n_total // world
    lo = rank * n_local
    W2 = 2 * L64
    REC = W2 + 1

    # ---- synthetic inputs (SURVEY 8d): bases with known discrete logs generated on the device,
    # uniform canonical scalars generated on the host (numpy PCG64, rejection-sampled below r)
    a0, dstep = 0x1234567, 0x89ABCDE
    d_bases = torch.empty((n_local, W2), dtype=torch.int64, device=dev)
    _lib.check(L.zkm_testgen_progression_device(CURVE_ID, 1, a0 + lo * dstep, dstep, n_local,
                                                ctypes.c_void_p(d_bases.data_ptr()), sp))
    torch.cuda.synchronize()
    reg = zkm.RegisteredBases.from_device(CURVE_ID, 1, d_bases.data_ptr(), n_local)
    del d_bases
    from oracle import capi  # input generator + checker only
    h_scal = torch.from_numpy(capi.random_scalars(CURVE_ID, n_local, seed=0x5EED0000 + LOG_N + 1000 * rank)
                              .view(np.int64)).pin_memory()
    d_scal = h_scal.to(dev)
    d_rec = torch.zeros(REC, dtype=torch.int64, device=dev)
    d_all = torch.zeros((world, REC), dtype=torch.int64, device=dev)
    d_final = torch.zeros(REC, dtype=torch.int64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        reg.msm_device(d_scal.data_ptr(), n_local, d_rec.data_ptr(), stream=stream)
        if world > 1:
            dist.all_gather_into_tensor(d_all.view(-1), d_rec)
            _lib.check(L.zkm_points_sum_device(CURVE_ID, 1, ctypes.c_void_p(d_all.data_ptr()), world,
                                               ctypes.c_void_p(d_final.data_ptr()), sp))

    h_out = np.zeros(W2, dtype=np.uint64)
    h_inf = np.zeros(1, dtype=np.uint8)
    h_rec = torch.zeros(REC, dtype=torch.int64).pin_memory()

    def step_e2e():
        """Host buffers in, host result out, through the C ABI."""
        if world == 1:
            _lib.check(L.zkm_msm_registered(reg.handle, 0, ctypes.c_void_p(h_scal.data_ptr()), n_local,
                                            ctypes.c_void_p(h_out.ctypes.data), ctypes.c_void_p(h_inf.ctypes.data)))
        else:
            d_s = h_scal.to(dev, non_blocking=True)
            reg.msm_device(d_s.data_ptr(), n_local, d_rec.data_ptr(), stream=stream)
            dist.all_gather_into_tensor(d_all.view(-1), d_rec)
            _lib.check(L.zkm_points_sum_device(CURVE_ID, 1, ctypes.c_void_p(d_all.data_ptr()), world,
                                               ctypes.c_void_p(d_final.data_ptr()), sp))
            h_rec.copy_(d_final, non_blocking=True)
            torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3 / steps
        ms = e0.elapsed_time(e1) / steps
        t = torch.tensor([ms, wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    # ---- headline: device-resident MSM
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(args.warmup):
        step_device()
    barrier()
    _lib.launch_count(reset=True)
    if sampler:
        sampler.start()
    ms_dev, _ = timed(step_device, args.steps, 0)
    clocks = sampler.stop() if sampler else None
    launches = _lib.launch_count()

    # ---- correctness of what was timed: known-discrete-log identity (exact big-int check on rank 0)
    final = (d_final if world > 1 else d_rec).cpu().numpy().view(np.uint64)
    dumps = {}      # --dump-outputs: name -> float64 array of the last timed step's outputs (u64 limbs as exact u32 words)
    if args.dump_outputs:
        dumps["msm_result_xy"] = final[:W2].view(np.uint32).astype(np.float64).reshape(2, -1)
        dumps["msm_result_infinity"] = final[W2:].astype(np.float64)
    ok = None
    if rank == 0:
        from oracle.py import exact
        from oracle.py.params import CURVES_BY_ID
        curve = CURVES_BY_ID[CURVE_ID]
        k = 0
        for r in range(world):      # every rank's scalars are reproducible from its seed
            sr = h_scal.numpy().view(np.uint64) if r == 0 else \
                capi.random_scalars(CURVE_ID, n_local, seed=0x5EED0000 + LOG_N + 1000 * r)
            s = sr.astype(object)
            sv = s[:, 0] + (s[:, 1] << 64) + (s[:, 2] << 128) + (s[:, 3] << 192)
            k += int(np.sum(sv * (a0 + (r * n_local + np.arange(n_local, dtype=object)) * dstep)))
        k %= curve.fr.modulus
        G = exact.Group(curve, 1)
        b, f = exact.point_to_bytes(curve, 1, G.mul(G.gen, k))
        ok = bool(final[W2] == f and final[:W2].tobytes() == b)

    # ---- stage breakdown + roofline of the dominant kernel (rank 0's slice)
    zkm.set_option("profile", 1)
    stages = np.zeros(6, dtype=np.float64)
    acc = np.zeros(6, dtype=np.float64)
    cnt = np.zeros(16, dtype=np.uint64)
    for _ in range(args.steps):
        reg.msm_device(d_scal.data_ptr(), n_local, d_rec.data_ptr(), stream=stream)
        _lib.check(L.zkm_profile_last_msm(ctypes.c_void_p(stages.ctypes.data)))
        acc += stages
    _lib.check(L.zkm_profile_last_msm_counts(ctypes.c_void_p(cnt.ctypes.data)))
    zkm.set_option("profile", 0)
    acc /= args.steps
    # bucket accumulation = batched-affine pair levels (k_pair_fwd / k_inv_batch / k_pair_bwd) + XYZZ tail
    accum_ms = float(acc[1] + acc[3])
    c_bits = zkm.msm_window_bits(CURVE_ID, 1, n_local)
    bits = 255 if CURVE_ID == 0 else 254
    windows = (bits + 1 + c_bits - 1) // c_bits    # signed digits: one spare bit for the carry
    algo_mads = ALGO_MODMULS_PER_POINT * n_local * MADS_PER_MODMUL
    # EXECUTED field products of the stage, from the device's own counters (zkm_profile_last_msm_counts -- exact list
    # sizes read back after the run, not estimates) and the per-operation product counts of the kernels' formulas:
    #   pairwise level : 6 per affine addition (1 in k_pair_fwd: run * d; 5 in k_pair_bwd: run * pre, run * d,
    #                    num * dinv, lambda^2, lambda * (x0 - x3)); pairs of a level = inputs - outputs;
    #                    + 3 per thread total and 1 per inversion thread in k_inv_batch (prefix, two unwind products, R^3)
    #   XYZZ tail      : 10 per mixed addition (madd-2008-s: 8M + 2S); the first entry of a task only loads
    entries, n_lvl, tasks = int(cnt[3]), int(cnt[12]), int(cnt[13])
    m_pair, m_inv = 64, 32                           # library defaults (options msm_pair_m / msm_pair_m2)
    lvl_in, products, pairs_total = entries, 0, 0
    for l in range(n_lvl):
        lvl_out = int(cnt[4 + l])
        pairs = lvl_in - lvl_out
        n_t = -(-lvl_out // m_pair)
        products += 6 * pairs + 3 * n_t + -(-n_t // m_inv)
        pairs_total += pairs
        lvl_in = lvl_out
    madds = max(lvl_in - tasks, 0)
    products += 10 * madds
    executed_mads = products * MADS_PER_MODMUL
    achieved = executed_mads / (accum_ms * 1e-3) / 1e9
    algo_rate = algo_mads / (accum_ms * 1e-3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        if tj.get("workload") == "%s_g1_msm_2p%d" % (CURVE_NAME, LOG_N) and world == 1:
            traffic = tj.get("bucket_accumulation_dram_bytes")
    except Exception:
        pass
    roofline = {
        "kernel": "bucket accumulation: k_pair_fwd/k_inv_batch/k_pair_bwd (batched-affine levels) + k_accum_affine (XYZZ tail)",
        "bound": "int_pipe",
        "achieved": achieved, "peak": IMAD_PEAK_GMADS, "unit": "GMAD/s", "frac": achieved / IMAD_PEAK_GMADS,
        "traffic": traffic, "kernel_ms": accum_ms,
        "executed": {"field_products": products, "wide_mads": executed_mads, "list_entries": entries, "affine_levels": n_lvl,
                     "affine_additions": pairs_total, "xyzz_mixed_additions": madds, "mads_per_product": MADS_PER_MODMUL,
                     "source": "zkm_profile_last_msm_counts (device counters of this run) x per-formula product counts"},
        "algorithmic": {"wide_mads": algo_mads, "gmads": algo_rate, "over_peak": algo_rate / IMAD_PEAK_GMADS,
                        "definition": "SURVEY 8d canonical count: 160 Fq products/point (16 windows x 10 per XYZZ mixed add) x "
                                      "%d wide MADs x %d points" % (MADS_PER_MODMUL, n_local),
                        "note": "exceeds the executed work (fewer windows at c=%d, 6-product affine additions with batched "
                                "inversion), so it can exceed the pipe peak; `frac` is the executed work" % c_bits},
        "peak_source": "measured: %s (profiles/int_pipe_peak_r2.jsonl, this pool's B200)" % IMAD_PEAK_SRC,
    }

    # ---- end to end through the host API
    ms_e2e, wall_e2e = timed(step_e2e, args.steps, 2)
    e2e = {"value": wall_e2e, "unit": "ms", "h2d_bytes_per_step": int(n_local * 32 * world),
           "d2h_bytes_per_step": int(REC * 8), "device_ms": ms_e2e,
           "note": "zkm_msm_registered: scalars from pinned host memory each step, affine result read back; bases "
                   "(the proving key) registered once; wall clock, max over ranks"}

    # ---- the same MSM over bases registered WITH precomputed window multiples (proving keys / SRS are
    # static: one-time table of W x the bases, all windows share one bucket set, no Horner tail).  Reported
    # beside the headline, not as the headline: `value` stays the plain registration.
    pre = None
    if not args.skip_precompute:
        d_b2 = torch.empty((n_local, W2), dtype=torch.int64, device=dev)
        _lib.check(L.zkm_testgen_progression_device(CURVE_ID, 1, a0 + lo * dstep, dstep, n_local,
                                                    ctypes.c_void_p(d_b2.data_ptr()), sp))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reg_pre = zkm.RegisteredBases.from_device(CURVE_ID, 1, d_b2.data_ptr(), n_local, precompute=True)
        torch.cuda.synchronize()
        reg_s = time.perf_counter() - t0
        if world == 1:
            # the literal multi_scalar_mul(bases, scalars) signature (zkm_msm_g1): HOST bases and HOST scalars.  The first
            # call uploads the bases (cold); later calls find them in the registration cache (fingerprint of 512 sampled
            # records per call) -- the proving key is the same vector for every proof (benches/groth16.rs:107-115).
            h_bases = d_b2.cpu().pin_memory()
            _lib.check(L.zkm_msm_cache_clear())
            cold = []
            for _ in range(4):
                t1 = time.perf_counter()
                _lib.check(L.zkm_msm_g1(CURVE_ID, ctypes.c_void_p(h_bases.data_ptr()), ctypes.c_void_p(0),
                                        ctypes.c_void_p(h_scal.data_ptr()), n_local, ctypes.c_void_p(h_out.ctypes.data),
                                        ctypes.c_void_p(h_inf.ctypes.data)))
                cold.append((time.perf_counter() - t1) * 1e3)
            e2e["unregistered_first_call_ms"] = cold[0]
            e2e["unregistered_ms"] = min(cold[1:])
            e2e["unregistered_over_registered"] = min(cold[1:]) / wall_e2e
            e2e["unregistered_h2d_bytes_first_call"] = int(n_local * (32 + W2 * 8))
            e2e["unregistered_same_result"] = bool(h_out.tobytes() == final[:W2].tobytes())
            zkm.set_option("msm_cache", 0)
            t1 = time.perf_counter()
            _lib.check(L.zkm_msm_g1(CURVE_ID, ctypes.c_void_p(h_bases.data_ptr()), ctypes.c_void_p(0),
                                    ctypes.c_void_p(h_scal.data_ptr()), n_local, ctypes.c_void_p(h_out.ctypes.data),
                                    ctypes.c_void_p(h_inf.ctypes.data)))
            e2e["unregistered_no_cache_ms"] = (time.perf_counter() - t1) * 1e3
            zkm.set_option("msm_cache", 1)
            _lib.check(L.zkm_msm_cache_clear())
            del h_bases
        del d_b2

        def step_pre():
            reg_pre.msm_device(d_scal.data_ptr(), n_local, d_rec.data_ptr(), stream=stream)
            if world > 1:
                dist.all_gather_into_tensor(d_all.view(-1), d_rec)
                _lib.check(L.zkm_points_sum_device(CURVE_ID, 1, ctypes.c_void_p(d_all.data_ptr()), world,
                                                   ctypes.c_void_p(d_final.data_ptr()), sp))
        ms_pre, _ = timed(step_pre, args.steps, 2)
        final_pre = (d_final if world > 1 else d_rec).cpu().numpy().view(np.uint64)
        pre = {"ms": ms_pre, "register_s": reg_s, "same_result_as_headline": bool(np.array_equal(final_pre, final)),
               "note": "bases registered with ZKM_REG_PRECOMPUTE (table of 2^(c w) P_i, W x the base memory)"}
        reg_pre.release()

    # ---- secondary headline: 2^24 Fr NTT (independent transform per GPU)
    ntt = None
    if not args.skip_ntt:
        n_ntt = 1 << LOG_N
        x = torch.from_numpy(capi.random_field_elements(CURVE_ID, n_ntt, seed=0x5EED1000 + LOG_N).view(np.int64)).to(dev)
        y = torch.empty_like(x)
        def step_ntt():
            _lib.check(L.zkm_ntt_device(CURVE_ID, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), LOG_N,
                                        0, 0, sp))
        ms_ntt, _ = timed(step_ntt, args.steps, 3)
        if args.dump_outputs:
            rows = np.sort(np.random.Generator(np.random.PCG64(0x5EED2000 + LOG_N)).choice(n_ntt, min(n_ntt, 1 << 16),
                                                                                          replace=False))
            dumps["ntt_sample_index"] = rows.astype(np.float64)
            dumps["ntt_sample_output"] = (y[torch.from_numpy(rows).to(dev)].cpu().numpy().view(np.uint32)
                                          .astype(np.float64))
        peaks = read_peaks()
        hbm = peaks["hbm_gbs"] if peaks and "hbm_gbs" in peaks else 6650.0
        gbs = 64.0 * n_ntt / (ms_ntt * 1e-3) / 1e9
        ntt_traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            if CURVE_ID == 0 and LOG_N == 24:
                ntt_traffic = tj.get("ntt_2p24_dram_bytes")
        except Exception:
            pass
        # integer-pipe view of the same kernel: (log2 n / 2) Fr products per element x 136 wide MADs
        ntt_mads = 0.5 * LOG_N * n_ntt * 136
        ntt_gmads = ntt_mads / (ms_ntt * 1e-3) / 1e9
        # end to end: pinned HOST buffer in and out through zkm_ntt (512 MiB each way at 2^24: PCIe-bound)
        h_x = torch.from_numpy(capi.random_field_elements(CURVE_ID, n_ntt, seed=0x5EED1000 + LOG_N).view(np.int64)).pin_memory()
        want_head = None
        def step_ntt_e2e():
            _lib.check(L.zkm_ntt(CURVE_ID, ctypes.c_void_p(h_x.data_ptr()), LOG_N, 0, 0))
        h_times = []
        for it in range(4):
            t1 = time.perf_counter()
            step_ntt_e2e()
            h_times.append((time.perf_counter() - t1) * 1e3)
        ntt_e2e = {"value": min(h_times[1:]), "unit": "ms", "h2d_bytes_per_step": int(n_ntt * 32), "d2h_bytes_per_step": int(n_ntt * 32),
                   "note": "zkm_ntt on a pinned host buffer, in place: upload, transform, download (wall clock, best of 3 after a "
                           "warm-up call)"}
        del h_x
        ntt_cpu = None
        if rank == 0 and world == 1 and not args.skip_cpu:
            ntt_cpu = cpu_ntt_baseline(LOG_N)
        ntt = {"metric": "Fr NTT 2^%d ms (%s)" % (LOG_N, CURVE_NAME), "ms": ms_ntt,
               "e2e": ntt_e2e, "cpu_baseline": ntt_cpu,
               "ntts_per_s_all_gpus": world * 1e3 / ms_ntt,
               "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s",
                            "algorithmic": "64 B/element (read once + write once)", "traffic": ntt_traffic},
               "int_pipe": {"achieved": ntt_gmads, "peak": IMAD_PEAK_GMADS, "unit": "GMAD/s",
                            "frac": ntt_gmads / IMAD_PEAK_GMADS,
                            "algorithmic": "log2(n)/2 Fr products per element x 136 wide MADs, the nominal 2 N^2 + N of an 8-limb "
                                           "Montgomery product (executed: + the four-step and coset products, ~1 per element per "
                                           "extra pass; BLS12-381 Fr issues 120 per product: its reduction limbs p_0 = 1 and "
                                           "p_1 = 2^32 - 1 need no multiplication)",
                            "executed_mads_per_product": 120 if CURVE_NAME == "bls12_381" else 136,
                            "peak_source": "measured: %s (profiles/int_pipe_peak_r2.jsonl)" % IMAD_PEAK_SRC},
               "note": "device-resident, out of place; integer-pipe bound on B200 (see DESIGN.md): the HBM fraction "
                       "is reported as the contract asks, int_pipe is the binding roofline"}
        del x, y

    # ---- third headline of BASELINE.json's metric: Groth16 proofs/s.  A zkMember-shaped PROXY (MSM + NTT
    # work of create_proof at domain 2^16; tools/groth16_proxy.py) run on every GPU as an independent
    # replica (batched proofs are distributed per GPU, no collective); the per-GPU rates are summed.
    proxy = None
    if not args.skip_proxy:
        torch.cuda.synchronize()
        cmd = [sys.executable, os.path.join(ROOT, "tools", "groth16_proxy.py"), "--log-n", "16", "--proofs", "160",
               "--inflight", "4", "--device", str(local_rank)]
        if world > 1:
            cmd += ["--host-wait", "2"]      # replicas share the host's cores: block instead of spinning on the read-back
        if rank == 0 and world == 1 and not args.skip_cpu:
            cmd.append("--cpu")
        try:
            env = dict(os.environ)
            for k in ("RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
                env.pop(k, None)
            outp = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
            mine = json.loads(outp.stdout.strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001
            mine = {"error": repr(e)}
        rates = torch.tensor([mine.get("proofs_per_s", 0.0)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(rates, op=dist.ReduceOp.SUM)
        proxy = dict(mine)
        proxy["proofs_per_s_all_gpus"] = float(rates[0])
        proxy["replicas"] = world

    # ---- the other bench configurations of BASELINE.json, rank 0 at N = 1 only (sub-objects, not the headline):
    # the Marlin-shaped proxy (config 4: KZG10 commits + transforms of one Marlin::prove) and the Groth16 proxy on
    # BW6-761, the second curve benches/groth16.rs instantiates.
    extra = {}
    if rank == 0 and world == 1 and not args.skip_proxy:
        def run_tool(name, cmd):
            try:
                outp = subprocess.run([sys.executable, os.path.join(ROOT, "tools", cmd[0])] + cmd[1:], capture_output=True,
                                      text=True, timeout=600)
                extra[name] = json.loads(outp.stdout.strip().splitlines()[-1])
            except Exception as e:  # noqa: BLE001
                extra[name] = {"error": repr(e)}
        torch.cuda.synchronize()
        run_tool("marlin_proxy", ["marlin_proxy.py", "--log-h", "16", "--log-k", "18", "--proofs", "6"]
                 + ([] if args.skip_cpu else ["--cpu"]))
        run_tool("groth16_proxy_bw6_761", ["groth16_proxy.py", "--curve", "bw6_761", "--log-n", "16", "--proofs", "48",
                                           "--inflight", "4"])

    # ---- one PROCESS driving all N GPUs through the C ABI (the Rust prover is a single process: zkm_init_mask +
    # ZKM_REG_SHARD; per-device host threads, partial sums gathered over NVLink P2P and added on device 0).  Rank 0 only,
    # after the per-rank measurements; the other ranks wait at the barrier below with their GPUs idle.
    single = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)           # every rank has finished its own GPU work: the GPUs are idle from here on
    if world > 1 and rank == 0 and not args.skip_single_process:
        try:
            reg.release()
            zkm.shutdown()
            zkm.init(list(range(world)))
            Ls = _lib.lib()
            d_all_b = torch.empty((n_total, W2), dtype=torch.int64, device=dev)
            _lib.check(Ls.zkm_testgen_progression_device(CURVE_ID, 1, a0, dstep, n_total, ctypes.c_void_p(d_all_b.data_ptr()), sp))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            reg_all = zkm.RegisteredBases.from_device(CURVE_ID, 1, d_all_b.data_ptr(), n_total, shard=True)
            reg_s = time.perf_counter() - t0
            del d_all_b
            h_all = torch.cat([h_scal] + [torch.from_numpy(capi.random_scalars(CURVE_ID, n_local, seed=0x5EED0000 + LOG_N + 1000 * r)
                                                           .view(np.int64)) for r in range(1, world)]).pin_memory()
            ts = []
            for it in range(2 + args.steps):
                t1 = time.perf_counter()
                _lib.check(Ls.zkm_msm_registered(reg_all.handle, 0, ctypes.c_void_p(h_all.data_ptr()), n_total,
                                                 ctypes.c_void_p(h_out.ctypes.data), ctypes.c_void_p(h_inf.ctypes.data)))
                if it >= 2:
                    ts.append((time.perf_counter() - t1) * 1e3)
            single = {"e2e_ms": sum(ts) / len(ts), "e2e_ms_best": min(ts), "gpus": world, "register_s": reg_s,
                      "same_result_as_headline": bool(h_out.tobytes() == final[:W2].tobytes() and int(h_inf[0]) == int(final[W2])),
                      "note": "ONE process, zkm_init_devices(0..N-1), bases registered with ZKM_REG_SHARD, zkm_msm_registered with "
                              "all 2^%d host scalars: upload of each shard's slice, N pipelines, P2P gather of N records, "
                              "k_points_sum on device 0, read-back (wall clock)" % LOG_N}
            reg_all.release()
            zkm.shutdown()
        except Exception as e:  # noqa: BLE001
            single = {"error": repr(e)}
    if world > 1:
        dist.barrier(group=cpu_group)

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        cpu = cpu_baseline_run(1, CPU_LOG_N)

    if rank == 0:
        line = {
            "metric": METRIC, "value": ms_dev, "unit": "ms", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32-limb Montgomery integers (381-bit Fq, 255-bit Fr)", "data": "synthetic",
            "config": {"workload": "G1 MSM, %s, 2^%d points total (range-sharded %d-way), uniform canonical scalars, "
                                   "bases (a0+i*d)*G" % (CURVE_NAME, LOG_N, world),
                       "window_bits": c_bits, "windows": windows, "l2": "inputs larger than L2 (scalars %d MiB + bases "
                       "%d MiB per GPU)" % (n_local * 32 >> 20, n_local * W2 * 8 >> 20),
                       "result_check": "known-discrete-log identity over all ranks' inputs, exact big-int",
                       "result_ok": ok},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "msm_stage_ms": {"sort": acc[0], "affine_levels": acc[1], "tasks": acc[2], "accumulate_xyzz": acc[3], "fold": acc[4], "reduce": acc[5]},
            "cpu_baseline": cpu, "ntt": ntt, "groth16_proxy": proxy, "msm_precomputed_bases": pre,
            "single_process_multi_gpu": single,
        }
        line.update(extra)
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0 if (ok is None or ok) else 2


if __name__ == "__main__":
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner on stdout) and anything
    # else written to fd 1 during the run go to stderr instead; the line itself is written to the saved descriptor.
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    import io
    _buf = io.StringIO()
    _orig = sys.stdout
    sys.stdout = _buf
    _rc = 1
    try:
        _rc = main()
    finally:
        sys.stdout = _orig
        _lines = [l for l in _buf.getvalue().splitlines() if l.strip()]
        _json = [l for l in _lines if l.lstrip().startswith("{")]
        for l in _lines:
            if l not in _json[-1:]:
                sys.stderr.write(l + "\n")
        if _json:
            os.write(_real_stdout, (_json[-1] + "\n").encode())
        os.close(_real_stdout)
    sys.exit(_rc)
