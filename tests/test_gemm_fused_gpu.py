"""The fused projections of the tcgen05 forward schedule through the C ABI, each against fp64 torch:
Gram-generating GEMM (K1 -> linear_g1 fusion), [X P^T | gd] projection, grouped launch."""
import pytest
import torch

pytestmark = pytest.mark.gpu
TOL = 2e-5


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()


def split(w):
    from sgrl_b200._lib import lib, ptr, stream, check
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    check(lib.sgrl_split_tf32(ptr(w), ptr(hi), ptr(lo), w.numel(), stream()), "split")
    return hi, lo


def fold(W):
    """(N,1024) -> triangle-folded (N,544), csrc/layout.h"""
    from sgrl_b200.packing import pack_indices
    slots, ri, ci = pack_indices()
    W3 = W.reshape(W.shape[0], 32, 32)
    Wf = torch.zeros(W.shape[0], 544, dtype=W.dtype, device=W.device)
    ri_t, ci_t = torch.tensor(ri, device=W.device), torch.tensor(ci, device=W.device)
    Wf[:, slots] = torch.where(ri_t == ci_t, W3[:, ri, ci], W3[:, ri, ci] + W3[:, ci, ri])
    return Wf


@pytest.mark.parametrize("T,N,keep", [(2304, 256, 1), (300, 128, 0), (1000, 256, 1), (129, 256, 0)])
def test_gram_gemm(T, N, keep):
    from sgrl_b200._lib import lib, ptr, stream, check
    g = torch.Generator(device="cuda").manual_seed(T + N)
    Z = torch.randn(T, 3, 32, device="cuda", generator=g)
    Z[:, :, 30] = torch.tensor([0.0, 0.0, -9.81], device="cuda")
    W = torch.randn(N, 1024, device="cuda", generator=g) / 32.0
    b = torch.randn(N, device="cuda", generator=g)
    Wf = fold(W).contiguous()
    hi, lo = split(Wf)
    Cm = torch.full((T, N + 4), 7.0, device="cuda")
    F = torch.zeros(T, device="cuda")
    Gp = torch.full((T, 544), 3.0, device="cuda") if keep else None
    check(lib.sgrl_gemm_gram(ptr(Z), ptr(hi), ptr(lo), ptr(b), ptr(Cm), N + 4, ptr(F), ptr(Gp), T, N, 1, stream()), "gram")
    torch.cuda.synchronize()
    Zd = Z.double()
    G = Zd.transpose(1, 2) @ Zd                                  # (T,32,32)
    ref = torch.relu(G.reshape(T, 1024) @ W.double().T + b.double())
    assert rel(Cm[:, :N], ref) < TOL
    assert torch.all(Cm[:, N:] == 7.0)
    assert rel(F, G.reshape(T, -1).norm(dim=1) + 1.0) < 1e-6
    if keep:
        from sgrl_b200.packing import pack_indices, tri_table
        slots, ri, ci = pack_indices()
        pads = [p for p, e in enumerate(tri_table()) if e is None]
        assert rel(Gp[:, slots], G[:, ri, ci]) < 1e-6 and torch.all(Gp[:, pads] == 0)


@pytest.mark.parametrize("T,N", [(40000, 256), (38001, 128), (60000, 256)])
def test_gram_gemm_persistent(T, N):
    """Persistent GRAM projection of inference passes (csrc/gemm_tc_persist.cuh: all N <= 256 columns in one tile, every packed Gram
    row generated once) against fp64 and against the per-tile kernel, each selected by the persist override of sgrl_gemm_desc;
    row tail, sub-matrix ldc, F = ||G|| + 1."""
    from gpu_util import gemm_desc
    from sgrl_b200.packing import GP_K
    g = torch.Generator(device="cuda").manual_seed(T + N)
    Z = torch.randn(T, 3, 32, device="cuda", generator=g)
    Z[:, :, 30] = torch.tensor([0.0, 0.0, -9.81], device="cuda")
    W = torch.randn(N, 1024, device="cuda", generator=g) / 32.0
    b = torch.randn(N, device="cuda", generator=g)
    hi, lo = split(fold(W).contiguous())
    out = []
    for persist in (1, 0):
        Cm = torch.full((T, N + 4), 7.0, device="cuda")
        F = torch.zeros(T, device="cuda")
        plan = gemm_desc(persist, A=None, gram_z=Z, gram_f=F, B=hi, B_hi=hi, B_lo=lo, ldb=GP_K, C=Cm, ldc=N + 4, M=T, N=N, K=GP_K,
                         bias=b, relu=1)
        assert plan["path"] == 2 and plan["gram"] == 1 and plan["persist"] == persist, plan
        out.append((Cm, F))
    Zd = Z.double()
    G = Zd.transpose(1, 2) @ Zd
    ref = torch.relu(G.reshape(T, 1024) @ W.double().T + b.double())
    for Cm, F in out:
        assert rel(Cm[:, :N], ref) < TOL
        assert torch.all(Cm[:, N:] == 7.0)
        assert rel(F, G.reshape(T, -1).norm(dim=1) + 1.0) < 1e-6
    assert torch.equal(out[0][1], out[1][1])                      # F: same products and summation order in both kernels


@pytest.mark.parametrize("T3,K,ldw", [(6912, 128, 128), (900, 128, 136), (601, 128, 128)])
def test_gd_projection(T3, K, ldw):
    from sgrl_b200._lib import lib, ptr, stream, check
    g = torch.Generator(device="cuda").manual_seed(T3)
    T = T3 // 3
    T3 = T * 3
    X = torch.randn(T3, K, device="cuda", generator=g)
    Wfull = torch.randn(40, ldw, device="cuda", generator=g) / K ** 0.5      # rows 30.. stand for the next tensors of the arena
    gd = torch.randn(T, 3, 2, device="cuda", generator=g)
    hi, lo = split(Wfull)
    Z = torch.full((T3, 32), 5.0, device="cuda")
    check(lib.sgrl_gemm_gd(ptr(X), K, ptr(hi), ptr(lo), ldw, ptr(gd), ptr(Z), T3, K, stream()), "gd")
    torch.cuda.synchronize()
    ref = torch.cat([X.double() @ Wfull[:30, :K].double().T, gd.reshape(T3, 2).double()], dim=1)
    assert rel(Z, ref) < TOL
    assert torch.equal(Z[:, 30:], gd.reshape(T3, 2))


@pytest.mark.parametrize("s0,s1", [((2304, 128, 256), (6912, 252, 128)), ((2304, 128, 256), (2304, 1024, 256)), ((300, 768, 256), (900, 30, 128))])
def test_grouped_pair(s0, s1):
    from sgrl_b200._lib import lib, ptr, stream, check
    g = torch.Generator(device="cuda").manual_seed(s0[0] + s1[1])
    ops = []
    for M, N, K in (s0, s1):
        A = torch.randn(M, K, device="cuda", generator=g)
        W = torch.randn(N + 2, K, device="cuda", generator=g) / K ** 0.5
        b = torch.randn(N, device="cuda", generator=g)
        ldc = (N + 7) // 4 * 4
        ops.append((A, W, b, torch.full((M, ldc), 2.0, device="cuda"), ldc, M, N, K) + split(W))
    a, c = ops
    check(lib.sgrl_gemm_pair(ptr(a[0]), a[7], ptr(a[8]), ptr(a[9]), ptr(a[2]), ptr(a[3]), a[4], a[5], a[6], a[7],
                             ptr(c[0]), c[7], ptr(c[8]), ptr(c[9]), ptr(c[2]), ptr(c[3]), c[4], c[5], c[6], c[7], 1, stream()), "pair")
    torch.cuda.synchronize()
    for A, W, b, Cm, ldc, M, N, K, _, _ in ops:
        ref = torch.relu(A.double() @ W[:N].double().T + b.double())
        assert rel(Cm[:, :N], ref) < TOL
        assert torch.all(Cm[:, N:] == 2.0)
