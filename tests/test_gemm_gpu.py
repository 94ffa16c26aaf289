"""K3 projections through the C ABI: fp32 SIMT kernel and the tcgen05 3xTF32 kernel vs fp64 torch.
Covers the three contraction forms of the hot path (Y=XW^T, dX=dYW, dW=dY^T X), ragged tails,
sub-matrix leading dimensions and the fused epilogue options the ABI exposes."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


def run_gemm(A, lda, ta, B, ldb, tb, Cm, ldc, M, N, K, alpha=1.0, bias=None, rowdiv=None, relu=0, acc=0, splitk=1, use_tc=0):
    from sgrl_b200._lib import lib, ptr, stream, check
    check(lib.sgrl_gemm(ptr(A), lda, ta, ptr(B), ldb, tb, ptr(Cm), ldc, M, N, K, alpha, ptr(bias), ptr(rowdiv), relu, acc, splitk, use_tc, stream()), "sgrl_gemm")
    torch.cuda.synchronize()


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


TOL = {0: 2e-6, 1: 2e-5}   # tcgen05 accumulates with truncation: ~5e-6 at K=1024, still 20x inside the 1e-4 budget
FWD = [(300, 256, 1024), (2304, 768, 256), (77, 252, 128), (128, 128, 32), (1000, 1024, 256), (129, 130, 100),
       (9, 256, 544), (27, 252, 128), (1, 1024, 256), (32, 130, 148), (16, 3, 256)]   # M <= 32: the skinny kernel of B=1..3 rollouts


@pytest.mark.parametrize("use_tc", [0, 1])
@pytest.mark.parametrize("M,N,K", FWD)
def test_forward_linear(use_tc, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    ldk = (K + 3) // 4 * 4
    X = torch.randn(M, ldk, device="cuda", generator=g)
    W = torch.randn(N, ldk, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    F = torch.rand(M, device="cuda", generator=g) * 500 + 100
    if use_tc and M * N * K < (1 << 21):
        pytest.skip("below the tcgen05 eligibility threshold (launch-bound sizes stay on the SIMT kernel)")
    Y = torch.full((M, N + 3), 7.0, device="cuda")                    # ldc > N: neighbours must stay untouched
    run_gemm(X, ldk, 0, W, ldk, 0, Y, N + 3, M, N, K, bias=b, rowdiv=F, relu=1, use_tc=use_tc)
    ref = torch.relu(X[:, :K].double() @ W[:, :K].double().T + b.double()) / F.double()[:, None]
    assert rel(Y[:, :N], ref) < TOL[use_tc]
    assert torch.all(Y[:, N:] == 7.0)


@pytest.mark.parametrize("use_tc", [0, 1])
@pytest.mark.parametrize("M,Nw,Kw", [(900, 768, 256), (2700, 252, 128), (600, 256, 1024), (2700, 30, 128)])
def test_data_gradient(use_tc, M, Nw, Kw):
    g = torch.Generator(device="cuda").manual_seed(Nw)
    ldn = (Nw + 3) // 4 * 4 if Nw != 30 else 32
    dY = torch.randn(M, ldn, device="cuda", generator=g)
    W = torch.randn(Nw, Kw, device="cuda", generator=g)
    dX = torch.randn(M, Kw, device="cuda", generator=g)
    base = dX.clone()
    run_gemm(dY, ldn, 0, W, Kw, 1, dX, Kw, M, Kw, Nw, acc=1, use_tc=use_tc)       # dX += dY W
    ref = base.double() + dY[:, :Nw].double() @ W.double()
    assert rel(dX, ref) < TOL[use_tc]


@pytest.mark.parametrize("use_tc", [0, 1])
@pytest.mark.parametrize("T,Nw,Kw,splitk", [(900, 256, 1024, 3), (2304, 1024, 256, 4), (6912, 128, 256, 8), (700, 30, 128, 2), (333, 512, 256, 1)])
def test_weight_gradient(use_tc, T, Nw, Kw, splitk):
    g = torch.Generator(device="cuda").manual_seed(T)
    ldn = (Nw + 3) // 4 * 4 if Nw != 30 else 32
    dY = torch.randn(T, ldn, device="cuda", generator=g)
    X = torch.randn(T, Kw, device="cuda", generator=g)
    dW = torch.zeros(Nw, Kw, device="cuda")
    run_gemm(dY, ldn, 1, X, Kw, 1, dW, Kw, Nw, Kw, T, alpha=0.5, acc=1, splitk=splitk, use_tc=use_tc)   # dW += 0.5 dY^T X
    ref = 0.5 * dY[:, :Nw].double().T @ X.double()
    assert rel(dW, ref) < TOL[use_tc]


def test_tc_rejects_unaligned_operands():
    from sgrl_b200._lib import SgrlError
    X = torch.randn(256, 145, device="cuda"); W = torch.randn(128, 145, device="cuda"); Y = torch.empty(256, 128, device="cuda")
    with pytest.raises(SgrlError, match="tcgen05"):
        run_gemm(X, 145, 0, W, 145, 0, Y, 128, 256, 128, 145, use_tc=1)
    run_gemm(X, 145, 0, W, 145, 0, Y, 128, 256, 128, 145, use_tc=0)
    assert rel(Y, X.double() @ W.double().T) < 2e-6


@pytest.mark.parametrize("M,N,K,tb", [(300, 256, 1024, 0), (2304, 768, 256, 0), (77, 252, 128, 0), (900, 256, 768, 1), (2700, 128, 252, 1), (600, 1024, 256, 1)])
def test_presplit_weights(M, N, K, tb):
    """tcgen05 path with the weight operand pre-split into tf32 hi/lo arenas (sgrl_split_tf32): Y = X W^T (tb=0) and
    dX = dY W (tb=1, W is (K,N) row-major read MN-major)."""
    from sgrl_b200._lib import lib, ptr, stream, check
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    X = torch.randn(M, K, device="cuda", generator=g)
    W = (torch.randn(N, K, device="cuda", generator=g) if not tb else torch.randn(K, N, device="cuda", generator=g)) / K ** 0.5
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    check(lib.sgrl_split_tf32(ptr(W), ptr(hi), ptr(lo), W.numel(), stream()))
    assert torch.all((hi.view(torch.int32) & 0x1FFF) == 0) and torch.all((lo.view(torch.int32) & 0x1FFF) == 0)
    assert rel(hi.double() + lo.double(), W) < 3e-7
    b = torch.randn(N, device="cuda", generator=g)
    Y = torch.full((M, N + 4), 7.0, device="cuda")
    check(lib.sgrl_gemm_presplit(ptr(X), K, 0, ptr(hi), ptr(lo), W.shape[1], tb, ptr(Y), N + 4, M, N, K, 1.0, ptr(b), None, 0, 0, 1, stream()))
    torch.cuda.synchronize()
    ref = X.double() @ (W.double().T if not tb else W.double()) + b.double()
    assert rel(Y[:, :N], ref) < TOL[1]
    assert torch.all(Y[:, N:] == 7.0)


@pytest.mark.parametrize("M,N,K,rowdiv,relu", [(40000, 768, 256, 1, 0), (38017, 252, 128, 0, 0), (40000, 128, 256, 0, 1), (37990, 1024, 384, 1, 1),
                                               (150000, 512, 256, 0, 1)])
def test_persistent_projection_kernel(M, N, K, rowdiv, relu):
    """Persistent inference variant (csrc/gemm_tc_persist.cuh: tile loop per SM, two accumulator buffers, TMA tensor stores) against
    fp64: row / column tails, the /F + column-scale and relu epilogues, sub-matrix ldc with untouched neighbours, more tiles than
    two rounds of the 148 SMs; and against the per-tile kernel, each selected by the persist override of sgrl_gemm_desc."""
    from sgrl_b200._lib import lib, ptr, stream, check
    from gpu_util import gemm_desc
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    X = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    check(lib.sgrl_split_tf32(ptr(W), ptr(hi), ptr(lo), W.numel(), stream()))
    b = torch.randn(N, device="cuda", generator=g)
    F = torch.rand(M, device="cuda", generator=g) * 500 + 100

    def run(persist):
        Y = torch.full((M, N + 4), 7.0, device="cuda")
        plan = gemm_desc(persist, A=X, lda=K, B=hi, B_hi=hi, B_lo=lo, ldb=K, C=Y, ldc=N + 4, M=M, N=N, K=K, bias=b,
                         rowdiv=F if rowdiv else None, relu=relu)
        assert plan["path"] == 2 and plan["persist"] == persist, plan
        return Y
    n0 = lib.sgrl_launch_count()
    Y = run(1)
    assert lib.sgrl_launch_count() == n0 + 1
    ref = X.double() @ W.double().T + b.double()
    if relu:
        ref = torch.relu(ref)
    if rowdiv:
        ref = ref / F.double()[:, None]
    assert rel(Y[:, :N], ref) < TOL[1]
    assert torch.all(Y[:, N:] == 7.0)
    Y2 = run(0)
    assert rel(Y2[:, :N], ref) < TOL[1] and rel(Y[:, :N], Y2[:, :N]) < 1e-5


@pytest.mark.parametrize("N", [64, 128, 512])
def test_update_shapes_against_fp64(N):
    """The tcgen05 kernel at the 2 304-row shapes of a B=256 humanoid update, against fp64 torch: forward projection against
    pre-split weights, data gradient (pre-split B read MN-major), weight gradient (both operands MN-major, split on the fly)
    and the Gram-generating projection."""
    from sgrl_b200._lib import lib, ptr, stream, check
    from sgrl_b200.packing import pack_indices
    g = torch.Generator(device="cuda").manual_seed(N)
    M, K = 2304, 256
    X = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    check(lib.sgrl_split_tf32(ptr(W), ptr(hi), ptr(lo), W.numel(), stream()))
    b = torch.randn(N, device="cuda", generator=g)
    F = torch.rand(M, device="cuda", generator=g) * 500 + 100
    dY = torch.randn(M, N, device="cuda", generator=g)
    Z = torch.randn(M, 3, 32, device="cuda", generator=g)
    Wf = torch.randn(N, 544, device="cuda", generator=g) / 23.0
    fhi, flo = torch.empty_like(Wf), torch.empty_like(Wf)
    check(lib.sgrl_split_tf32(ptr(Wf), ptr(fhi), ptr(flo), Wf.numel(), stream()))
    Y = torch.zeros(M, N, device="cuda")
    check(lib.sgrl_gemm_presplit(ptr(X), K, 0, ptr(hi), ptr(lo), K, 0, ptr(Y), N, M, N, K, 1.0, ptr(b), ptr(F), 1, 0, 1, stream()))
    dX = torch.zeros(M, K, device="cuda")        # dX = dY W: B = W (N,K) read "transposed"
    check(lib.sgrl_gemm_presplit(ptr(dY), N, 0, ptr(hi), ptr(lo), K, 1, ptr(dX), K, M, K, N, 1.0, None, None, 0, 0, 1, stream()))
    dW = torch.zeros(N, K, device="cuda")        # dW = dY^T X: both operands read "transposed"
    check(lib.sgrl_gemm(ptr(dY), N, 1, ptr(X), K, 1, ptr(dW), K, N, K, M, 1.0, None, None, 0, 1, 2, 1, stream()))   # splitk > 1: "may be split" (no cluster split-K)
    C = torch.zeros(M, N, device="cuda")
    Fo = torch.zeros(M, device="cuda")
    check(lib.sgrl_gemm_gram(ptr(Z), ptr(fhi), ptr(flo), ptr(b), ptr(C), N, ptr(Fo), None, M, N, 1, stream()))
    torch.cuda.synchronize()
    assert rel(Y, torch.relu(X.double() @ W.double().T + b.double()) / F.double()[:, None]) < TOL[1]
    assert rel(dX, dY.double() @ W.double()) < TOL[1]
    assert rel(dW, dY.double().T @ X.double()) < TOL[1]
    Zd = Z.double()
    G = Zd.transpose(1, 2) @ Zd                  # (M,32,32); the kernel generates its packed upper triangle (csrc/layout.h)
    slots, ri, ci = pack_indices()
    Gp = torch.zeros(M, 544, dtype=torch.float64, device="cuda")
    Gp[:, slots] = G[:, ri, ci]
    assert rel(C, torch.relu(Gp @ Wf.double().T + b.double())) < TOL[1]
    assert rel(Fo, G.reshape(M, -1).norm(dim=1) + 1.0) < 1e-6
