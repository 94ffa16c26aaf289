#!/usr/bin/env python
"""Device time of one pre-split tcgen05 projection (K-major operands), CUDA events over `reps` back-to-back launches.
usage: gemm_time.py M N K [rowdiv] [reps]   (the plan the library's tile model picks for the shape)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sgrl_b200._lib import lib, ptr, stream, check

M, N, K = (int(x) for x in sys.argv[1:4])
reps = int(sys.argv[5]) if len(sys.argv) > 5 else 20
X = torch.randn(M, K, device="cuda")
W = torch.randn(N, K, device="cuda")
hi, lo = torch.empty_like(W), torch.empty_like(W)
check(lib.sgrl_split_tf32(ptr(W), ptr(hi), ptr(lo), W.numel(), stream()))
Y = torch.empty(M, N, device="cuda")
rowdiv = len(sys.argv) > 4 and sys.argv[4] == "1"
F = torch.rand(M, device="cuda") * 900 + 100 if rowdiv else None


gram = len(sys.argv) > 6 and sys.argv[6] == "gram"      # A generated from Z (K = 544 packed Gram rows): M N 544 0 reps gram
if gram:
    Z = torch.randn(M, 96, device="cuda")
    Fo = torch.zeros(M, device="cuda")


def run():
    if gram:
        check(lib.sgrl_gemm_gram(ptr(Z), ptr(hi), ptr(lo), None, ptr(Y), N, ptr(Fo), None, M, N, 1, stream()))
        return
    check(lib.sgrl_gemm_presplit(ptr(X), K, 0, ptr(hi), ptr(lo), K, 0, ptr(Y), N, M, N, K, 1.0, None, ptr(F) if rowdiv else None, 0, 0, 1, stream()))


for _ in range(3):
    run()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    run()
e1.record()
torch.cuda.synchronize()
us = e0.elapsed_time(e1) * 1e3 / reps
ref = X[:4096].double() @ W.double().t()
if gram:
    ref = Y[:4096].double()      # checked in tests/test_gemm_fused_gpu.py
if rowdiv:
    ref = ref / F[:4096].double()[:, None]
err = ((Y[:4096].double() - ref).norm() / ref.norm()).item()
print(f"GEMM {M}x{N}x{K}{' /F' if rowdiv else ''}: {us:8.1f} us  {2.0 * M * N * K / us * 1e-6:7.1f} TFLOP/s  rel err {err:.1e}  [{' '.join(k + '=' + v for k, v in sorted(os.environ.items()) if k.startswith('SGRL_'))}]")
