"""Fixed-base batch scalar multiplication sweep (zkm_fixed_base_msm*): one JSONL row per (curve, group, n).

    python tools/fixed_base_sweep.py --out profiles/sweep_fixed_base_r4.jsonl [--quick]

  device_ms       CUDA events around zkm_fixed_base_msm_device, scalars resident in HBM, median of --reps after one
                  warm-up call of the same shape (table build + scalar kernel + normalisation: the whole call)
  e2e_ms          zkm_fixed_base_msm with pinned host buffers (upload, the same kernels, download), median of --reps
  outputs_per_s   n / device_ms
  check           weighted-sum identity on that row's outputs: sum r_i out_i (variable-base MSM, another kernel path)
                  == (sum r_i s_i mod r) B (one exact multiplication), r_i random 64-bit
One more row, "groth16_setup_2p20": the six batches of a 2^20-constraint proving key (a, b_g1, b_g2, h, l,
gamma_abc_g1) issued one after another through the host entry point, as ark-groth16's generator issues them.
The first row records the GPU name and power limit of the run.  A CPU figure is not measured here.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.py import exact  # noqa: E402
from oracle.py.params import BLS12_381, BN254, BW6_761  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # the row still says what it could not read
        return {"gpu": "unknown (%s)" % e}


def rand_mont(curve, n, seed):
    S, bits = curve.fr.limbs64, curve.fr.bits
    rng = np.random.Generator(np.random.PCG64(seed))
    m = rng.integers(0, 1 << 64, size=(n, S), dtype=np.uint64)
    m[:, S - 1] &= np.uint64((1 << (bits - 1 - 64 * (S - 1))) - 1)
    return m


def weighted_sum_mod_r(curve, m, rw):
    r, S = curve.fr.modulus, m.shape[1]
    m16 = m.view(np.uint16).reshape(len(m), 4 * S).astype(np.uint64)
    r16 = rw.view(np.uint16).reshape(len(rw), 4).astype(np.uint64)
    total = 0
    for lo in range(0, len(m), 1 << 20):
        mb, rb = m16[lo:lo + (1 << 20)], r16[lo:lo + (1 << 20)]
        for a in range(4):
            sums = (rb[:, a:a + 1] * mb).sum(axis=0, dtype=np.uint64)
            total += sum(int(v) << (16 * (a + k)) for k, v in enumerate(sums))
    return total * pow(1 << (64 * S), -1, r) % r


def pinned(torch, shape, dtype):
    t = torch.empty(shape, dtype=dtype, pin_memory=True)
    return t, t.numpy()


def one_row(zkm, torch, curve, g, n, reps, seed):
    L = zkm.load()
    G = exact.Group(curve, g)
    rng = random.Random(seed)
    B = G.mul(G.gen, rng.randrange(2, curve.fr.modulus))
    base = np.frombuffer(exact.point_to_bytes(curve, g, B)[0], dtype=np.uint64).copy()
    W2 = base.size
    S = curve.fr.limbs64
    m = rand_mont(curve, n, seed)
    # device-resident leg, on a stream of our own: stream 0 would mean the library's own stream (include/zkm_b200.h),
    # which the events below would not see
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_s = torch.from_numpy(m.view(np.int64)).cuda()
        d_xy = torch.empty((n, W2), dtype=torch.int64, device="cuda")
        d_inf = torch.empty(n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    bp = ctypes.c_void_p(base.ctypes.data)

    def dev_call():
        zkm._lib.check(L.zkm_fixed_base_msm_device(curve.curve_id, g, bp, 0, ctypes.c_void_p(d_s.data_ptr()), n,
                                                   ctypes.c_void_p(d_xy.data_ptr()), ctypes.c_void_p(d_inf.data_ptr()),
                                                   ctypes.c_void_p(stream.cuda_stream)))
    dev_call()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        dev_call()
        e1.record(stream)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    device_ms = float(np.median(times))
    # host leg, pinned buffers
    _, h_s = pinned(torch, (n, S), torch.int64)
    h_s[:] = m.view(np.int64)
    _, h_xy = pinned(torch, (n, W2), torch.int64)
    _, h_inf = pinned(torch, (n,), torch.uint8)
    p = lambda a: ctypes.c_void_p(a.ctypes.data)

    def host_call():
        zkm._lib.check(L.zkm_fixed_base_msm(curve.curve_id, g, bp, 0, p(h_s), n, p(h_xy), p(h_inf)))
    host_call()
    et = []
    for _ in range(reps):
        t0 = time.perf_counter()
        host_call()
        et.append((time.perf_counter() - t0) * 1e3)
    e2e_ms = float(np.median(et))
    xy = h_xy.view(np.uint64)
    same = bool(np.array_equal(d_xy.cpu().numpy().view(np.uint64), xy) and np.array_equal(d_inf.cpu().numpy(), h_inf))
    # weighted-sum identity on the outputs
    rw = np.random.Generator(np.random.PCG64(seed + 1)).integers(0, 1 << 64, size=n, dtype=np.uint64)
    rsc = np.zeros((n, S), dtype=np.uint64)
    rsc[:, 0] = rw
    lhs = zkm.VariableBaseMSM.multi_scalar_mul(xy, rsc, curve=curve.name, group=g, infinity=h_inf)
    rhs = G.mul(B, weighted_sum_mod_r(curve, m, rw))
    want_xy, want_inf = exact.point_to_bytes(curve, g, rhs)
    check = bool(same and lhs.xy.tobytes() == want_xy and int(lhs.infinity) == want_inf)
    del d_s, d_xy, d_inf
    torch.cuda.empty_cache()
    return {"curve": curve.name, "group": g, "n": n, "log_n": int(np.log2(n)), "device_ms": round(device_ms, 4),
            "e2e_ms": round(e2e_ms, 3), "outputs_per_s": round(n / (device_ms * 1e-3)), "reps": reps,
            "device_equals_host": same, "check": check}


def groth16_setup_row(zkm, torch, reps, log_n=20, num_inputs=2):
    """The six fixed-base batches of circuit_specific_setup for a 2^log_n-constraint circuit with ~2^log_n variables."""
    C = BLS12_381
    nv = 1 << log_n
    sizes = [("a_query", 1, nv), ("b_g1_query", 1, nv), ("b_g2_query", 2, nv), ("h_query", 1, (1 << log_n) - 1),
             ("l_query", 1, nv - num_inputs), ("gamma_abc_g1", 1, num_inputs)]
    from oracle import capi
    bases = {1: capi.generator_mont(C.curve_id, 1), 2: capi.generator_mont(C.curve_id, 2)}
    bufs = []
    for k, (name, g, n) in enumerate(sizes):
        m = rand_mont(C, n, 0x6E0 + k)
        _, h_s = pinned(torch, (n, 4), torch.int64)
        h_s[:] = m.view(np.int64)
        W2 = bases[g].size
        bufs.append((name, g, n, h_s, pinned(torch, (n, W2), torch.int64)[1], pinned(torch, (n,), torch.uint8)[1]))
    L = zkm.load()
    p = lambda a: ctypes.c_void_p(a.ctypes.data)

    def run():
        per = {}
        for name, g, n, h_s, h_xy, h_inf in bufs:
            t0 = time.perf_counter()
            zkm._lib.check(L.zkm_fixed_base_msm(C.curve_id, g, p(bases[g]), 0, p(h_s), n, p(h_xy), p(h_inf)))
            per[name] = round((time.perf_counter() - t0) * 1e3, 3)
        return per
    run()
    runs = [run() for _ in range(reps)]
    total = [sum(r.values()) for r in runs]
    k = int(np.argsort(total)[len(total) // 2])
    # each batch: spot-check 8 outputs against the exact group law
    ok = True
    for name, g, n, h_s, h_xy, h_inf in bufs:
        G = exact.Group(C, g)
        rinv = pow(1 << 256, -1, C.fr.modulus)
        for i in random.Random(7).sample(range(n), min(8, n)):
            s = capi.limbs_to_ints(h_s[i:i + 1].view(np.uint64))[0] * rinv % C.fr.modulus
            xy, inf = exact.point_to_bytes(C, g, G.mul(G.gen, s) if s else None)
            ok &= h_xy[i].view(np.uint64).tobytes() == xy and int(h_inf[i]) == inf
    return {"row": "groth16_setup_2p20", "curve": C.name, "batches": {nm: n for nm, _, n in sizes}, "e2e_ms": round(total[k], 3),
            "per_batch_ms": runs[k], "reps": reps, "check": bool(ok)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="2^16 .. 2^18 only (rehearsal)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fixed_base_sweep: no CUDA device (the sweep measures the GPU; there is nothing to fall back to)")
    import zkmember_b200 as zkm
    zkm.init(0)
    info = gpu_info()
    rows = []
    plan = []
    for curve in (BLS12_381, BN254, BW6_761):
        for g in (1, 2):
            top = 24 if (curve is BLS12_381 and g == 1) else 22
            if a.quick:
                top = 18
            plan += [(curve, g, lg) for lg in range(16, top + 1)]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for i, (curve, g, lg) in enumerate(plan):
            row = one_row(zkm, torch, curve, g, 1 << lg, a.reps, 0x5EED + 97 * lg + 13 * g + curve.curve_id)
            if i == 0:
                row.update(info)
            rows.append(row)
            f.write(json.dumps(row) + "\n")
            f.flush()
            print(json.dumps(row), flush=True)
        if not a.quick:
            row = groth16_setup_row(zkm, torch, a.reps)
            row.update(info)
            f.write(json.dumps(row) + "\n")
            print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
