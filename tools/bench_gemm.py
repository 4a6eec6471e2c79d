#!/usr/bin/env python
"""Micro-benchmark of the tensor-core GEMM kernels at the shapes of the update path (CUDA events, inputs >> L2).
Usage: python tools/bench_gemm.py [--rows 1572864] [--reps 5]"""
import argparse
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from magpo_b200 import _lib as L  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=128 * 4096 * 3)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--only", default="")
args = ap.parse_args()
dev = torch.device("cuda:0")
M = args.rows
s = L.stream_ptr()
peak = 6539.9


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


print(f"rows={M}")
for (K, N) in [(64, 64), (64, 128), (64, 192), (64, 256), (128, 128), (128, 384), (256, 64), (192, 64), (384, 128)]:
    if args.only and args.only != "nn":
        break
    X = torch.randn(M, K, device=dev)
    WT = torch.randn(N, K, device=dev) * 0.1
    W = WT.t().contiguous()
    scr = torch.zeros(2 * N * K, device=dev)
    Y = torch.zeros(M, N, device=dev)
    ms_tc = timeit(lambda: L.call("magpo_test_gemm_tc", s, C.c_int64(M), N, K, L.ptr(X), K, L.ptr(WT), L.ptr(scr), None, L.ptr(Y), N, 0))
    ms_simt = timeit(lambda: L.call("magpo_test_gemm", s, 0, C.c_int64(M), N, K, L.ptr(X), L.ptr(W), None, L.ptr(Y), 0))
    gb = M * (K + N) * 4 / 1e9
    tf = 2.0 * M * N * K / 1e12
    print(f"NN K={K:3d} N={N:3d}: tcgen05 {ms_tc:7.3f} ms  {gb / ms_tc * 1e3:7.0f} GB/s ({gb / ms_tc * 1e3 / peak:4.2f} of HBM)  {tf / ms_tc * 1e3:6.1f} TF/s"
          f" | SIMT {ms_simt:7.3f} ms {tf / ms_simt * 1e3:6.1f} TF/s")
    del X, Y
for (K, N) in [(64, 64), (64, 128), (64, 256), (128, 128), (128, 384)]:
    if args.only and args.only != "tn":
        break
    X = torch.randn(M, K, device=dev)
    dY = torch.randn(M, N, device=dev)
    dW = torch.zeros(K, N, device=dev)
    ms_tc = timeit(lambda: L.call("magpo_test_gemm_tc_tn", s, C.c_int64(M), N, K, L.ptr(X), K, L.ptr(dY), N, L.ptr(dW), N))
    gb = M * (K + N) * 4 / 1e9
    tf = 2.0 * M * N * K / 1e12
    print(f"TN K={K:3d} N={N:3d}: tcgen05 {ms_tc:7.3f} ms  {gb / ms_tc * 1e3:7.0f} GB/s ({gb / ms_tc * 1e3 / peak:4.2f} of HBM)  {tf / ms_tc * 1e3:6.1f} TF/s")
    del X, dY
