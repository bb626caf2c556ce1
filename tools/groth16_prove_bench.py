"""Groth16 create_proof after synthesis: the one-call prover against the per-call paths it replaces.

    python tools/groth16_prove_bench.py --out profiles/groth16_prove_r5.jsonl [--proofs 24] [--quick]

One JSONL row per (curve, log_n, path, in_flight); the four paths alternate inside each configuration, one proof at a
time per host thread, `in_flight` threads:
  a_one_call    zkm_groth16_prove (zkmember_b200.groth16.create_proof): host a, b, c, assignment in, proof out
  b_per_call    what a Rust user gets without the prover fork: 7 host zkm_ntt calls (ifft + coset_fft of a, b, c, one
                coset_ifft; the pointwise step that upstream runs on the CPU between them is LEFT OUT, which only favours
                this path), 5 host zkm_msm_registered calls one after another, and the final assembly as four small host
                MSMs (the parent revision's _lincomb; upstream does it with arkworks on the CPU, which cannot run here:
                a stand-in, labelled as one)
  c_proxy_chain tools/groth16_proxy.py's device chain: zkm_witness_map_device, zkm_fr_into_repr_device and one
                zkm_msm_batch_registered_device on device-resident inputs, then one stream synchronise; NO assembly
  d_device_form zkm_groth16_prove_device on the same device-resident inputs as (c), then one stream synchronise: (c)
                plus the range check and the assembly.  (d) - (c) is what the assembly adds to a proof's critical path;
                (a) - (d) is the host side of (a): staging into the pinned buffer, the upload, the read-back
  proofs_per_s  proofs / wall time of the window;  latency_ms  median host call -> proof bytes (a, b) or -> records (c, d)
One more row per configuration, "assembly": device time per proof of k_g16_assemble_g1, k_g16_assemble_g2 and
k_g16_range.  The kernels run inside one library call, so their durations come from the CUDA activity records of a
torch.profiler run of its own (three device-form proofs), not from events of the timed windows.  The first row records
the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import capi  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # the row still says what it could not read
        return {"gpu": "unknown (%s)" % e}


def synthetic(cid, log_n, seed):
    """A key of zkMember's shape from progressions (known discrete logs), 50 % infinity in the b queries, witness-like
    assignment (45 % zero, 45 % one).  Returns (ProvingKey, kwargs of create_proof)."""
    from zkmember_b200.groth16 import ProvingKey
    n = 1 << log_n
    m, num_inputs = n - 5, 3
    num_aux = m - num_inputs
    rng = np.random.Generator(np.random.PCG64(seed))
    g1 = capi.progression(cid, 1, 3 + seed, 7, 3 * m + n + 8)
    g2 = capi.progression(cid, 2, 5 + seed, 11, m + 3)
    inf_b1 = (rng.random(m + 1) < 0.5).astype(np.uint8)
    inf_b2 = (rng.random(m + 1) < 0.5).astype(np.uint8)
    pk = ProvingKey(cid, g1[-1], g1[-2], g2[-1], g1[-3], g2[-2], g1[:m + 1], g1[m + 1:2 * m + 2], g2[:m + 1],
                    g1[2 * m + 2:2 * m + 1 + n], g1[2 * m + 1 + n:2 * m + 1 + n + num_aux],
                    infinity={"b_g1": inf_b1, "b_g2": inf_b2}, precompute=True)
    abc = [capi.random_field_elements(cid, n, seed=seed + k) for k in range(3)]
    full = capi.random_scalars(cid, m, seed=seed + 9, kind="witness")
    args = dict(r=int(rng.integers(1, 1 << 62)) ** 4, s=int(rng.integers(1, 1 << 62)) ** 4, a=abc[0], b=abc[1], c=abc[2],
                input_assignment=full[:num_inputs], aux_assignment=full[num_inputs:])
    return pk, args


def path_b(pk, args):
    """Per-call host path (see the module docstring)."""
    import ctypes
    from zkmember_b200 import _lib
    from zkmember_b200.msm import VariableBaseMSM, FR_WORDS
    from zkmember_b200.serialize import Proof, FR_MODULUS
    L = _lib.lib()
    cid = pk.curve
    S = FR_WORDS[cid]
    n = len(args["a"])
    log_n = n.bit_length() - 1
    vs = [np.array(args[k], copy=True) for k in ("a", "b", "c")]
    p = lambda x: ctypes.c_void_p(x.ctypes.data)
    for v in vs:
        _lib.check(L.zkm_ntt(cid, p(v), log_n, 1, 0))
        _lib.check(L.zkm_ntt(cid, p(v), log_n, 0, 1))
    h = vs[0]
    _lib.check(L.zkm_ntt(cid, p(h), log_n, 1, 1))
    from zkmember_b200.kzg import KZG10
    full = np.concatenate([args["input_assignment"], args["aux_assignment"]])
    h_acc = KZG10.commit(pk.msms.h, h[:n - 1])
    l_acc = pk.msms.l.msm(args["aux_assignment"])
    a_acc = pk.msms.a.msm(full)
    b1_acc = pk.msms.b_g1.msm(full)
    b2_acc = pk.msms.b_g2.msm(full)
    r, s = args["r"], args["s"]

    def lincomb(group, terms):
        xy = np.stack([t[0] for t in terms])
        inf = np.array([1 if t[1] else 0 for t in terms], dtype=np.uint8)
        sc = np.stack([np.array([((t[2] % FR_MODULUS[cid]) >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(S)], dtype=np.uint64)
                       for t in terms])
        return VariableBaseMSM.multi_scalar_mul(xy, sc, curve=cid, group=group, infinity=inf)
    g_a = lincomb(1, [(pk.delta_g1, False, r), (*pk.first["a"], 1), (a_acc.xy, a_acc.infinity, 1), (pk.alpha_g1, False, 1)])
    g1_b = lincomb(1, [(pk.delta_g1, False, s), (*pk.first["b_g1"], 1), (b1_acc.xy, b1_acc.infinity, 1), (pk.beta_g1, False, 1)])
    g2_b = lincomb(2, [(pk.delta_g2, False, s), (*pk.first["b_g2"], 1), (b2_acc.xy, b2_acc.infinity, 1), (pk.beta_g2, False, 1)])
    g_c = lincomb(1, [(g_a.xy, g_a.infinity, s), (g1_b.xy, g1_b.infinity, r), (pk.delta_g1, False, -(r * s)),
                      (l_acc.xy, l_acc.infinity, 1), (h_acc.xy, h_acc.infinity, 1)])
    return Proof(a=g_a, b=g2_b, c=g_c).serialize()


class ChainC:
    """groth16_proxy.py's device chain on resident inputs (one per host thread: its own buffers and stream)."""

    def __init__(self, pk, args):
        import torch
        from zkmember_b200.msm import coord_words
        self.pk, self.args = pk, args
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64).copy()).cuda()
        self.src = [dev(args[k]) for k in ("a", "b", "c")]
        self.abc = [torch.empty_like(x) for x in self.src]
        self.z = dev(np.concatenate([args["input_assignment"], args["aux_assignment"]]))
        W1, W2 = coord_words(pk.curve, 1), coord_words(pk.curve, 2)
        self.recs = [torch.zeros(2 * (2 * (W2 if k == 4 else W1) + 2), dtype=torch.int64, device="cuda") for k in range(5)]
        self.stream = torch.cuda.Stream()

    def run(self):
        import ctypes
        import torch
        from zkmember_b200 import _lib
        from zkmember_b200.msm import msm_batch_device, FR_WORDS
        L = _lib.lib()
        pk, cid = self.pk, self.pk.curve
        S = FR_WORDS[cid]
        n = len(self.args["a"])
        log_n = n.bit_length() - 1
        ni = len(self.args["input_assignment"])
        sp = ctypes.c_void_p(self.stream.cuda_stream)
        with torch.cuda.stream(self.stream):
            for d, s_ in zip(self.abc, self.src):
                d.copy_(s_)
            _lib.check(L.zkm_witness_map_device(cid, ctypes.c_void_p(self.abc[0].data_ptr()), ctypes.c_void_p(self.abc[1].data_ptr()),
                                                ctypes.c_void_p(self.abc[2].data_ptr()), log_n,
                                                ctypes.c_void_p(self.abc[1].data_ptr()), sp))
            _lib.check(L.zkm_fr_into_repr_device(cid, ctypes.c_void_p(self.abc[1].data_ptr()),
                                                 ctypes.c_void_p(self.abc[1].data_ptr()), pk.msms.h.n, sp))
            zp, m = self.z.data_ptr(), self.z.shape[0] // S
            ms = pk.msms
            msm_batch_device([(ms.b_g2, zp, m, self.recs[4].data_ptr()), (ms.h, self.abc[1].data_ptr(), ms.h.n, self.recs[0].data_ptr()),
                              (ms.l, zp + 8 * S * ni, ms.l.n, self.recs[1].data_ptr()), (ms.a, zp, m, self.recs[2].data_ptr()),
                              (ms.b_g1, zp, m, self.recs[3].data_ptr())], stream=self.stream.cuda_stream)
        self.stream.synchronize()


class ChainD(ChainC):
    """The device form on the same resident inputs as ChainC."""

    def __init__(self, pk, args):
        import torch
        from zkmember_b200.msm import coord_words
        super().__init__(pk, args)
        W1, W2 = coord_words(pk.curve, 1), coord_words(pk.curve, 2)
        self.out = torch.zeros(2 * (2 * W1 + 1) + 2 * W2 + 1 + 1, dtype=torch.int64, device="cuda")

    def run(self):
        import torch
        n = len(self.args["a"])
        with torch.cuda.stream(self.stream):
            for d, s_ in zip(self.abc, self.src):
                d.copy_(s_)
            self.pk.prove_device(self.abc[0].data_ptr(), self.abc[1].data_ptr(), self.abc[2].data_ptr(), n.bit_length() - 1,
                                 self.z.data_ptr(), len(self.args["input_assignment"]), self.args["r"], self.args["s"],
                                 self.out.data_ptr(), stream=self.stream.cuda_stream)
        self.stream.synchronize()


def window(fn_for_thread, in_flight, proofs):
    """proofs spread over in_flight host threads; returns (proofs/s, median latency ms)."""
    lat = []
    lock = threading.Lock()
    per = proofs // in_flight

    def worker(k):
        fn = fn_for_thread(k)
        for _ in range(per):
            t0 = time.perf_counter()
            fn()
            dt = (time.perf_counter() - t0) * 1e3
            with lock:
                lat.append(dt)
    th = [threading.Thread(target=worker, args=(k,)) for k in range(in_flight)]
    t0 = time.perf_counter()
    for t in th:
        t.start()
    for t in th:
        t.join()
    wall = time.perf_counter() - t0
    return per * in_flight / wall, statistics.median(lat)


def assembly_time(pk, args):
    """Device time of the assembly kernels per proof (torch.profiler, a run of its own)."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    chain = ChainD(pk, args)
    chain.run()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            chain.run()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.key_averages():
        for part in ("g16_assemble_g1", "g16_assemble_g2", "g16_range"):
            if "k_" + part in e.key:
                t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                tot[part] = tot.get(part, 0.0) + t / 1e3 / 3
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--proofs", type=int, default=24, help="proofs per timed window (a multiple of 4)")
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the four paths per configuration")
    ap.add_argument("--quick", action="store_true", help="log_n 12 only (a rehearsal)")
    a = ap.parse_args()
    import zkmember_b200 as zkm
    from zkmember_b200.groth16 import create_proof
    zkm.init(0)
    configs = [(0, 12)] if a.quick else [(0, 15), (0, 16), (2, 16)]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps({"row": "env", **gpu_info()}) + "\n")
        for cid, log_n in configs:
            pk, args = synthetic(cid, log_n, seed=60 + log_n)
            try:
                # path b leaves out the pointwise step (a cost stand-in): its h, hence its proof, differs; the proof
                # bytes of the one call against the per-call orchestration are pinned by tests/test_gpu_groth16_prove.py
                chains, dchains = {}, {}
                paths = {
                    "a_one_call": lambda k: (lambda: create_proof(pk, **args).serialize()),
                    "b_per_call": lambda k: (lambda: path_b(pk, args)),
                    "c_proxy_chain": lambda k: (chains[k] if k in chains else chains.setdefault(k, ChainC(pk, args))).run,
                    "d_device_form": lambda k: (dchains[k] if k in dchains else dchains.setdefault(k, ChainD(pk, args))).run,
                }
                for name in paths:      # warm every path and thread count once
                    for inf in (1, 4):
                        window(paths[name], inf, 4)
                res = {}
                for rnd in range(a.rounds):
                    for inf in (1, 4):
                        for name in paths:
                            res.setdefault((name, inf), []).append(window(paths[name], inf, a.proofs))
                for (name, inf), v in res.items():
                    row = {"row": "prove", "curve": ["bls12_381", "bn254", "bw6_761"][cid], "log_n": log_n, "path": name,
                           "in_flight": inf, "proofs_per_s": round(statistics.median([x[0] for x in v]), 1),
                           "latency_ms": round(statistics.median([x[1] for x in v]), 3),
                           "rounds": [[round(x[0], 1), round(x[1], 3)] for x in v]}
                    f.write(json.dumps(row) + "\n")
                    f.flush()
                    print(row, flush=True)
                asm = assembly_time(pk, args)
                row = {"row": "assembly", "curve": ["bls12_381", "bn254", "bw6_761"][cid], "log_n": log_n,
                       **{k + "_kernel_ms": round(v, 3) for k, v in sorted(asm.items())}}
                f.write(json.dumps(row) + "\n")
                print(row, flush=True)
            finally:
                pk.release()


if __name__ == "__main__":
    main()
