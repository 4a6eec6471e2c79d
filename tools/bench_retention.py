#!/usr/bin/env python
"""Micro-benchmark of the chunkwise tensor-core retention kernels at the update's shape."""
import argparse
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from magpo_b200 import _lib as L  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--T", type=int, default=128)
ap.add_argument("--N", type=int, default=4096)
ap.add_argument("--A", type=int, default=3)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
T, N, A = args.T, args.N, args.A
dev = torch.device("cuda:0")
torch.manual_seed(0)
pk = torch.randn(T, N, A, 256, device=dev) * 0.5
dpk = torch.zeros(T, N, A, 256, device=dev)
ret = torch.zeros(T, N, A, 64, device=dev)
dret = torch.randn(T, N, A, 64, device=dev)
Hs = torch.zeros(T, N, 64, 64, device=dev)
H0 = torch.randn(N, 64, 64, device=dev) * 0.3
Hout = torch.zeros(N, 64, 64, device=dev)
done = (torch.rand(T, N, device=dev) < 0.01).to(torch.uint8)
s = L.stream_ptr()
base, db = pk.data_ptr(), dpk.data_ptr()
tokens = T * N * A


def run(bwd, causal):
    if not bwd:
        L.call("magpo_test_retention", s, 0, T, N, A, C.c_float(0.775), causal, C.c_void_p(base), C.c_void_p(base + 256),
               C.c_void_p(base + 512), 256, L.ptr(H0), L.ptr(done), L.ptr(ret), L.ptr(Hs), L.ptr(Hout), None, None, None, None, 0)
    else:
        L.call("magpo_test_retention", s, 1, T, N, A, C.c_float(0.775), causal, C.c_void_p(base), C.c_void_p(base + 256),
               C.c_void_p(base + 512), 256, L.ptr(H0), L.ptr(done), None, L.ptr(Hs), None, L.ptr(dret), C.c_void_p(db),
               C.c_void_p(db + 256), C.c_void_p(db + 512), 256)


def timeit(fn):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.reps


print(f"T={T} N={N} A={A} tokens={tokens}")
for causal in (0, 1):
    run(0, causal)  # the backward reads the states of the matching forward
    f = timeit(lambda: run(0, causal))
    b = timeit(lambda: run(1, causal))
    fb, bb = tokens * 4 * 256, tokens * 7 * 256
    print(f"chunk causal={causal}: fwd {f:7.3f} ms ({fb / f / 1e6:7.0f} GB/s algorithmic)   "
          f"bwd {b:7.3f} ms ({bb / b / 1e6:7.0f} GB/s algorithmic)")
