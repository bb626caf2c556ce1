#!/usr/bin/env python3
"""MarlinKZG10 on the GPU at zkMember's Marlin shapes: the round commitments (nine polynomials, g_1 and g_2 with degree
bounds, so eleven items, hiding on) as one `zkm_kzg_commit_many` call, and the opening at beta and gamma as one
`zkm_kzg_open_batch` call (host form, host to host) and one `zkm_kzg_open_batch_device` call (CUDA events on the stream).
The SRS is a synthetic progression of D + 1 = 6 |K| + 1 points (known discrete logs), coefficients are uniform.

Also reported, alternating with the calls above on the same inputs:
  msm_only_ms   the same 2 x 2 MSMs alone (zkm_msm_batch_registered_device on resident canonical scalars): the MSM share;
                the rest of the device time is the O(n) kernels (combinations, divisions, evaluations, into_repr)
  proxy_open_ms the opening phase of tools/marlin_proxy.py, two concurrent hiding zkm_kzg_open calls of 3|H| and 6|K|
                coefficients: a lower bound, it does less work than MarlinKZG10
`check` is a linearity cross-check: the opening of all terms equals the group sum of the openings of two halves of the
terms (and random_v and the evaluations likewise), checked with exact arithmetic.  No CPU leg exists for MarlinKZG10 here.
Writes one JSON line per configuration to stdout (and to --out when given).

  python tools/marlin_pc_bench.py [--curve bls12_381|bw6_761] [--log-h 15] [--log-k 17] [--reps 5] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import random
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zkmember_b200 as zkm  # noqa: E402
from zkmember_b200 import _lib  # noqa: E402
from zkmember_b200.kzg import KZG10, Powers  # noqa: E402
from oracle import capi  # noqa: E402  (input generator / checker only)
from oracle.py import exact  # noqa: E402
from oracle.py.params import BLS12_381, BW6_761  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--curve", default="bls12_381", choices=["bls12_381", "bw6_761"])
ap.add_argument("--log-h", type=int, default=15)
ap.add_argument("--log-k", type=int, default=17)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", default=None)
args = ap.parse_args()

curve = {"bls12_381": BLS12_381, "bw6_761": BW6_761}[args.curve]
cid, fr = curve.curve_id, curve.fr
S, W = fr.limbs64, 2 * capi.coord_words(cid, 1)
H, K = 1 << args.log_h, 1 << args.log_k
D = 6 * K
zkm.init(0)
L = _lib.lib()
pg = Powers(cid, capi.progression(cid, 1, 11, 13, D + 1))
pgg = Powers(cid, capi.progression(cid, 1, 17, 19, D + 2))
rand = lambda n, seed: capi.random_field_elements(cid, n, seed=seed).reshape(-1, S)
arr = lambda ct, v: ctypes.cast((ct * max(len(v), 1))(*v), ctypes.c_void_p)
p_ = lambda a: ctypes.c_void_p(a.ctypes.data)

# round commitments: w, z_a, z_b, mask | t, g_1 (bound |H| - 2), h_1 | g_2 (bound |K| - 2), h_2   (hiding bound 1)
sizes = [H, H, H, 3 * H, 2 * H, H - 1, 2 * H, K - 1, 6 * K - 5]
bounded = {5: H - 2, 7: K - 2}
polys = [rand(n, 100 + i) for i, n in enumerate(sizes)]
items = []
for i, c in enumerate(polys):
    items.append((c, 0, rand(2, 200 + i)))
    if i in bounded:
        items.append((c, D - bounded[i], rand(2, 300 + i)))


def commit_many():
    k = len(items)
    out, inf = np.zeros((k, W), np.uint64), np.zeros(k, np.uint8)
    _lib.check(L.zkm_kzg_commit_many(pg.handle, pgg.handle, k, arr(ctypes.c_void_p, [c.ctypes.data for c, _, _ in items]),
                                     arr(ctypes.c_size_t, [len(c) for c, _, _ in items]), arr(ctypes.c_size_t, [s for _, s, _ in items]),
                                     arr(ctypes.c_void_p, [b.ctypes.data for _, _, b in items]), arr(ctypes.c_size_t, [2] * k), p_(out), p_(inf)))


# opening: beta with g_1 (and its shifted term), z_b, t, mask; gamma with g_2 (and shifted) and the inner LC (h_2, g_2)
blinds = [rand(2, 400 + i) for i in range(len(sizes))] + [rand(2, 500), rand(2, 501)]
xi = rand(12, 600)
zs = rand(2, 700)
terms = [(0, 5, 5, 0, 0), (0, 5, 9, D - bounded[5], 1), (0, 2, 2, 0, 2), (0, 4, 4, 0, 3), (0, 3, 3, 0, 4),
         (1, 7, 7, 0, 5), (1, 7, 10, D - bounded[7], 6), (1, 8, 8, 0, 7), (1, 7, 7, 0, 8)]


def open_args(ts):
    cols = [arr(ctypes.c_int32, [t[i] for t in ts]) for i in range(3)] + [arr(ctypes.c_size_t, [t[3] for t in ts])]
    tc = np.concatenate([xi[t[4]] for t in ts])
    return cols, tc


def open_host(ts, evals=True):
    cols, tc = open_args(ts)
    w, wi, rv = np.zeros((2, W), np.uint64), np.zeros(2, np.uint8), np.zeros((2, S), np.uint64)
    ev = np.zeros((len(ts), S), np.uint64)
    _lib.check(L.zkm_kzg_open_batch(pg.handle, pgg.handle, len(polys), arr(ctypes.c_void_p, [c.ctypes.data for c in polys]),
                                    arr(ctypes.c_size_t, [len(c) for c in polys]), len(blinds),
                                    arr(ctypes.c_void_p, [b.ctypes.data for b in blinds]), arr(ctypes.c_size_t, [2] * len(blinds)), 2,
                                    p_(zs), len(ts), *cols, p_(tc), p_(w), p_(wi), p_(rv), p_(ev) if evals else None))
    return w, wi, rv, ev


dev = lambda a: torch.from_numpy(a.view(np.int64).copy()).cuda()
dpolys, dblinds = [dev(c) for c in polys], [dev(b) for b in blinds]
dw = torch.zeros(2 * (W + 1), dtype=torch.int64, device="cuda")
drv = torch.zeros(2 * S, dtype=torch.int64, device="cuda")
dev_ = torch.zeros(len(terms) * S, dtype=torch.int64, device="cuda")
stream = torch.cuda.current_stream()
cols, tc = open_args(terms)


def open_device():
    _lib.check(L.zkm_kzg_open_batch_device(pg.handle, pgg.handle, len(polys), arr(ctypes.c_void_p, [t.data_ptr() for t in dpolys]),
                                           arr(ctypes.c_size_t, [len(c) for c in polys]), len(blinds),
                                           arr(ctypes.c_void_p, [t.data_ptr() for t in dblinds]), arr(ctypes.c_size_t, [2] * len(blinds)),
                                           2, p_(zs), len(terms), *cols, p_(tc), ctypes.c_void_p(dw.data_ptr()),
                                           ctypes.c_void_p(drv.data_ptr()), ctypes.c_void_p(dev_.data_ptr()),
                                           ctypes.c_void_p(stream.cuda_stream)))


# the four MSMs of the opening alone, on resident canonical scalars of the same lengths
wlen = [max(D - bounded[5] + H - 2, 3 * H - 1), max(D - bounded[7] + K - 2, 6 * K - 6)]
msm_sc = [dev(capi.random_scalars(cid, n, seed=800 + i)) for i, n in enumerate(wlen + [1, 1])]
msm_out = torch.zeros(4 * 128, dtype=torch.int64, device="cuda")


def msm_only():
    hs = [pg.handle, pg.handle, pgg.handle, pgg.handle]
    ns = wlen + [1, 1]
    _lib.check(L.zkm_msm_batch_registered_device(4, arr(ctypes.c_uint64, hs), arr(ctypes.c_size_t, [0] * 4),
                                                 arr(ctypes.c_void_p, [t.data_ptr() for t in msm_sc]), arr(ctypes.c_size_t, ns),
                                                 arr(ctypes.c_void_p, [msm_out.data_ptr() + 128 * 8 * i for i in range(4)]),
                                                 ctypes.c_void_p(stream.cuda_stream)))


px = [rand(3 * H, 900), rand(6 * K, 901)]


def proxy_open():
    th = [threading.Thread(target=KZG10.open, args=(pg, px[i], zs[i], pgg, blinds[i])) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def dev_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b)


legs = {"commit_many_ms": lambda: host_ms(commit_many), "open_batch_ms": lambda: host_ms(lambda: open_host(terms)),
        "open_batch_device_ms": lambda: dev_ms(open_device), "msm_only_ms": lambda: dev_ms(msm_only),
        "proxy_open_ms": lambda: host_ms(proxy_open)}
for fn in legs.values():      # warm-up of every shape
    fn()
times = {k: [] for k in legs}
for _ in range(args.reps):
    for k, fn in legs.items():
        times[k].append(fn())

# linearity cross-check: all terms == first half + second half
G = exact.Group(curve, 1)
pt = lambda w, wi, i: exact.point_from_bytes(curve, 1, w[i].tobytes(), int(wi[i]))
full, a, b = open_host(terms), open_host(terms[:4]), open_host(terms[4:])
r = fr.modulus
ints = lambda v: [fr.from_mont(x) for x in capi.limbs_to_ints(v)]
check = all(pt(full[0], full[1], i) == G.add(pt(a[0], a[1], i), pt(b[0], b[1], i)) for i in range(2))
check &= ints(full[2]) == [(x + y) % r for x, y in zip(ints(a[2]), ints(b[2]))]
check &= ints(full[3]) == ints(a[3]) + ints(b[3])
check &= np.array_equal(full[3], dev_.cpu().numpy().view(np.uint64).reshape(-1, S))
gpu = os.popen("nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader").read().strip()
row = {"curve": args.curve, "log_h": args.log_h, "log_k": args.log_k, "D": D, "items": len(items), "terms": len(terms),
       "reps": args.reps, "check": bool(check), "gpu": gpu}
for k, v in times.items():
    row[k] = round(float(np.median(v)), 3)
line = json.dumps(row)
print(line, flush=True)
if args.out:
    with open(args.out, "a") as f:
        f.write(line + "\n")
