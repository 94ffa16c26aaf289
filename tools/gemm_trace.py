#!/usr/bin/env python
"""Prints the SM-clock timeline of CTA 0 of one tcgen05 GEMM launch (sgrl_gemm_trace): prologue, TMA issue,
operand landing, split done, MMA issue, accumulator ready, epilogue done.  usage: gemm_trace.py M N K [pre] [tb] [mode]
mode: gram (A generated from Z, K = 544)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sgrl_b200._lib import lib, ptr, stream, check


def main():
    M, N, K = (int(x) for x in sys.argv[1:4])
    pre = len(sys.argv) > 4 and sys.argv[4] == "1"
    tb = int(sys.argv[5]) if len(sys.argv) > 5 else 0
    X = torch.randn(M, K, device="cuda")
    W = torch.randn(N, K, device="cuda") if not tb else torch.randn(K, N, device="cuda")
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    check(lib.sgrl_split_tf32(ptr(W), ptr(hi), ptr(lo), W.numel(), stream()))
    Y = torch.empty(M, N, device="cuda")
    buf = torch.zeros(64, dtype=torch.int64, device="cuda")

    mode = sys.argv[6] if len(sys.argv) > 6 else ""
    Z, F = torch.randn(M, 96, device="cuda"), torch.zeros(M, device="cuda")

    def run():
        if mode == "gram":
            check(lib.sgrl_gemm_gram(ptr(Z), ptr(hi), ptr(lo), None, ptr(Y), N, ptr(F), None, M, N, 0, stream()))
        elif pre:
            check(lib.sgrl_gemm_presplit(ptr(X), K, 0, ptr(hi), ptr(lo), W.shape[1], tb, ptr(Y), N, M, N, K, 1.0, None, None, 0, 0, 1, stream()))
        else:
            check(lib.sgrl_gemm(ptr(X), K, 0, ptr(W), W.shape[1], tb, ptr(Y), N, M, N, K, 1.0, None, None, 0, 0, 1, 1, stream()))
    for _ in range(5):
        run()
    torch.cuda.synchronize()
    lib.sgrl_gemm_trace(ptr(buf))
    run()
    torch.cuda.synchronize()
    lib.sgrl_gemm_trace(None)
    t = buf.cpu().tolist()
    t0 = t[0]
    rel = lambda i: (t[i] - t0) if t[i] else None
    print(f"# GEMM {M}x{N}x{K} pre={int(pre)} tb={tb} {mode}: cycles since CTA-0 entry")
    print("prologue done", rel(1), "| acc ready", rel(2), "| epilogue done", rel(3), "| all warps joined", rel(4))
    print("epilogue chunk 0: tmem loaded", rel(5), "| staged", rel(6), "| stored", rel(7), "| first store iterations", [rel(56 + i) for i in range(4)])
    for name, base in (("tma issued ", 8), ("full landed", 20), ("split done ", 32), ("mma issue  ", 44)):
        print(name, [rel(base + i) for i in range(12) if t[base + i]])


if __name__ == "__main__":
    main()
