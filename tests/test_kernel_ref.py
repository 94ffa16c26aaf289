"""The packed-layout fp64 references of tests/kernel_ref.py restate the oracle (and through it the reference,
subequivariant_attentions.py:90-151), not the kernels: fed the traced intermediates of oracle.set_oracle.transformer_model
in the token layout, they reproduce the traced outputs to rounding.  CPU only."""
import pytest
import torch

import kernel_ref as R
from oracle import set_oracle as O
from sgrl_b200 import graph as G, morphologies as M, synth

CASES = [("3d_humanoid_9_full", 3), ("3d_walker_2_right_leg_left_knee", 2), ("3d_cheetah_14_full", 2)]
TOL = 1e-12


def rel(a, b):
    return ((a - b).norm() / b.norm()).item()


def _trace(name, B, kind):
    par = M.ALL[name]
    N = len(par)
    g = G.build_graph(par)
    g64 = dict(g, relation=g["relation"].double())
    p = {k: v.double() for k, v in O.synth_params(kind, 7).items()}
    b = synth.make_batch(B, N, seed=3)
    x = b["obs"].view(B, N, 41).double()
    if kind == "critic":
        x = torch.cat([x, b["action"].view(B, N, 3).double()], 2)
    trace = {}
    with torch.no_grad():
        O.transformer_model(p, x, g64, trace=trace)
    return p, g64["relation"], N, trace


def _tok(t, T):
    """(B, N, ...) oracle tensor -> packed (T, per-token) rows."""
    return t.reshape(T, -1)


@pytest.mark.parametrize("name,B", CASES)
@pytest.mark.parametrize("kind", ["actor", "critic"])
def test_attention_ref_reproduces_oracle(name, B, kind):
    p, relation, N, tr = _trace(name, B, kind)
    T = B * N
    cu = torch.arange(B + 1, dtype=torch.int32) * N
    rw, rb = p["transformer_encoder.rel_encoder.weight"], p["transformer_encoder.rel_encoder.bias"]
    for l in range(3):
        bias = l == 0
        for rel_off in ((None, torch.zeros(B, dtype=torch.int32)) if bias else (None,)):
            o, og, pp = R.attention_fwd_ref(_tok(tr[f"{l}.QKV"], T), _tok(tr[f"{l}.VGP"], T), _tok(tr["GD"], T),
                                            rw if bias else None, rb if bias else None, cu, rel_off, relation.flatten())
            assert rel(o, _tok(tr[f"{l}.O"], T)) < TOL
            assert rel(og.reshape(T, -1), _tok(tr[f"{l}.OG"], T)) < TOL
            pref = torch.zeros(T, 2, 16, dtype=torch.float64)
            pref[..., :N] = tr[f"{l}.P"].reshape(T, 2, N)
            assert (pp - pref).abs().max().item() < TOL
            assert torch.all(pp[..., N:] == 0)


@pytest.mark.parametrize("name,B", CASES)
def test_inv_feature_ref_reproduces_oracle(name, B):
    p, _, N, tr = _trace(name, B, "actor")
    T = B * N
    gd = _tok(tr["GD"], T)
    pre = "transformer_encoder.layers.{}."
    for l in range(3):
        # layer input: one projection (g_proj); after the attention: two (g_proj2, g_proj3) of the same dV
        Z, Z2, Gp, F = R.inv_feature_fwd_ref(tr[f"{l}.VGIN"].reshape(T, 3, 128), None, gd,
                                             p[pre.format(l) + "self_attn.g_proj.weight"])
        assert Z2 is None
        _check_feature(Z, Gp, F, tr[f"{l}.Z1"], tr[f"{l}.G1"], tr[f"{l}.F1"], T)
        Z, Z2, Gp, F = R.inv_feature_fwd_ref(tr[f"{l}.DV"].reshape(T, 3, 128), None, gd,
                                             p[pre.format(l) + "g_proj2.weight"], p[pre.format(l) + "g_proj3.weight"])
        _check_feature(Z, Gp, F, tr[f"{l}.Z2"], tr[f"{l}.G2"], tr[f"{l}.F2"], T)
        assert rel(Z2, tr[f"{l}.Z3"].reshape(T, 3, 32)) < TOL
    # head: X = [v0 | Vg] (C = 136)
    Z, _, Gp, F = R.inv_feature_fwd_ref(tr["VGF"].reshape(T, 3, 128), tr["V0"].reshape(T, 3, 8), gd, p["gg_proj.weight"])
    _check_feature(Z, Gp, F, tr["ZH"], tr["GH"], tr["FH"], T)


def _check_feature(Z, Gp, F, Zr, Gr, Fr, T):
    from sgrl_b200.packing import pack_indices
    slots, ri, ci = pack_indices()
    full = Gr.reshape(T, 32, 32)
    assert rel(Z, Zr.reshape(T, 3, 32)) < TOL
    assert rel(Gp[:, slots], full[:, ri, ci]) < TOL
    pad = sorted(set(range(544)) - set(slots))
    assert len(pad) == 16 and torch.all(Gp[:, pad] == 0)
    assert rel(F, Fr.reshape(T)) < TOL


def test_inv_feature_bwd_ref_folded_convention():
    """dGp[p(i,j)] = dL/dG_ij + dL/dG_ji: the reference backward equals autograd of <D, G> over the full Gram for any D,
    ignores the padding slots, and matches a central finite difference at one token."""
    torch.manual_seed(0)
    from sgrl_b200.packing import pack_indices
    slots, ri, ci = pack_indices()
    T = 5
    Z = torch.randn(T, 3, 32, dtype=torch.float64)
    D = torch.randn(T, 32, 32, dtype=torch.float64)
    dF = torch.randn(T, dtype=torch.float64)
    ri_, ci_ = torch.tensor(ri), torch.tensor(ci)
    dGp = torch.full((T, 544), 1e3, dtype=torch.float64)          # garbage in the padding slots
    dGp[:, slots] = torch.where(ri_ == ci_, D[:, ri_, ci_], D[:, ri_, ci_] + D[:, ci_, ri_])
    dZ = R.inv_feature_bwd_ref(dGp, dF, Z)

    z = Z.clone().requires_grad_(True)
    G = z.transpose(-1, -2) @ z
    ((D * G).sum() + (dF * (torch.linalg.matrix_norm(G) + 1)).sum()).backward()
    assert rel(dZ, z.grad) < 1e-13

    def loss(zt):
        Gt, Gpt = R.gram_packed(zt[None])
        return (dGp[1, slots] * Gpt[0, slots]).sum() + dF[1] * (torch.linalg.matrix_norm(Gt[0]) + 1)
    h = 1e-6
    fd = torch.zeros(3, 32, dtype=torch.float64)
    for r in range(3):
        for c in range(32):
            e = torch.zeros(3, 32, dtype=torch.float64)
            e[r, c] = h
            fd[r, c] = (loss(Z[1] + e) - loss(Z[1] - e)) / (2 * h)
    assert rel(dZ[1], fd) < 1e-7

    # Z = 0: ||G|| has no gradient there; the convention (and the kernel) take the subgradient 0
    dz0 = R.inv_feature_bwd_ref(dGp[:1], dF[:1], torch.zeros(1, 3, 32, dtype=torch.float64))
    assert torch.all(dz0 == 0)


def test_attention_bwd_ref_finite_difference():
    """attention_bwd_ref against central differences of <d_o, o> + <d_og, og> on a ragged two-graph batch with a bias."""
    torch.manual_seed(1)
    cu = torch.tensor([0, 3, 5], dtype=torch.int32)
    T = 5
    qkv = torch.randn(T, 768, dtype=torch.float64) * 0.1
    vgp = torch.randn(T, 756, dtype=torch.float64)
    gd = torch.randn(T, 6, dtype=torch.float64)
    rw, rb = torch.randn(2, 3, dtype=torch.float64), torch.randn(2, dtype=torch.float64)
    relation = torch.randn(9 * 3 + 4 * 3, dtype=torch.float64)
    rel_off = torch.tensor([0, 27], dtype=torch.int32)
    do, dog = torch.randn(T, 256, dtype=torch.float64), torch.randn(T, 768, dtype=torch.float64)
    dq, dv, dw = R.attention_bwd_ref(qkv, vgp, gd, rw, rb, cu, rel_off, relation, do, dog)

    def L(q=qkv, v=vgp, w=rw):
        o, og, _ = R.attention_fwd_ref(q, v, gd, w, rb, cu, rel_off, relation)
        return (o * do).sum() + (og.reshape(T, -1) * dog).sum()
    h = 1e-6
    for (t, c) in ((0, 3), (2, 300), (4, 700), (3, 140)):
        e = torch.zeros_like(qkv)
        e[t, c] = h
        assert abs((L(q=qkv + e) - L(q=qkv - e)) / (2 * h) - dq[t, c]) < 1e-7
    for (t, c) in ((1, 5), (4, 755)):
        e = torch.zeros_like(vgp)
        e[t, c] = h
        assert abs((L(v=vgp + e) - L(v=vgp - e)) / (2 * h) - dv[t, c]) < 1e-7
    for hh in range(2):
        for c in range(3):
            e = torch.zeros_like(rw)
            e[hh, c] = h
            assert abs((L(w=rw + e) - L(w=rw - e)) / (2 * h) - dw[hh, c]) < 1e-7


def _gemm_problem(gen, M, N, K, nb, trans_a, trans_b, accumulate, epi):
    """Random SgrlGemmProblem of small size with every instance in its own slice of each flat buffer (z-strides padded)."""
    def buf(n):
        return torch.randn(n, generator=gen, dtype=torch.float64)
    lda, ldb, ldc = (M if trans_a else K) + 3, (N if trans_b else K) + 2, N + 5
    pr = dict(M=M, N=N, K=K, nb=nb, trans_a=trans_a, trans_b=trans_b, lda=lda, ldb=ldb, ldc=ldc, alpha=-0.75,
              accumulate=accumulate, relu="relu" in epi, colscale=1.5, colscale_n=3 if "colscale" in epi else 0,
              zs_a=(K if trans_a else M) * lda + 7, zs_b=(K if trans_b else N) * ldb + 1, zs_c=M * ldc + 2)
    pr["A"], pr["B"], pr["C"] = buf(nb * pr["zs_a"]), buf(nb * pr["zs_b"]), buf(nb * pr["zs_c"])
    pr["B_hi"] = None
    if "bias" in epi:
        pr["bias"], pr["zs_bias"] = buf(nb * (N + 1)), N + 1
    if "rowdiv" in epi:
        pr["rowdiv"], pr["zs_rowdiv"] = buf(nb * (M + 2)).abs() + 0.5, M + 2
    for k, ld in (("mask", "ldmask"), ("res1", "ldres1"), ("res2", "ldres2")):
        if k in epi:
            pr[ld] = N + 1
            pr[k], pr["zs_" + k] = buf(nb * M * (N + 1)), M * (N + 1)
    if "rowsum" in epi:
        pr["rowsum"], pr["zs_rowsum"] = buf(nb * (M + 3)), M + 3
    return pr


def _gemm_loop(pr):
    """gemm_simt_kernel's product and epilogue restated element by element (plain Python floats), and the fused row sum."""
    C, rs = pr["C"].clone(), (pr["rowsum"].clone() if pr.get("rowsum") is not None else None)
    M, N, K = pr["M"], pr["N"], pr["K"]
    for z in range(pr["nb"]):
        def A(m, k):
            return pr["A"][z * pr["zs_a"] + (k * pr["lda"] + m if pr["trans_a"] else m * pr["lda"] + k)].item()

        def B(n, k):
            return pr["B"][z * pr["zs_b"] + (k * pr["ldb"] + n if pr["trans_b"] else n * pr["ldb"] + k)].item()
        for m in range(M):
            if rs is not None:
                rs[z * pr["zs_rowsum"] + m] += pr["alpha"] * sum(A(m, k) for k in range(K))
            for n in range(N):
                v = pr["alpha"] * sum(A(m, k) * B(n, k) for k in range(K))
                if pr.get("bias") is not None:
                    v += pr["bias"][z * pr["zs_bias"] + n].item()
                if pr["relu"]:
                    v = max(v, 0.0)
                if pr.get("rowdiv") is not None:
                    v = v / pr["rowdiv"][z * pr["zs_rowdiv"] + m].item()
                if n < pr["colscale_n"]:
                    v *= pr["colscale"]
                if pr.get("mask") is not None:
                    v = v if pr["mask"][z * pr["zs_mask"] + m * pr["ldmask"] + n].item() > 0 else 0.0
                for r in ("res1", "res2"):
                    if pr.get(r) is not None:
                        v += pr[r][z * pr["zs_" + r] + m * pr["ld" + r] + n].item()
                c = z * pr["zs_c"] + m * pr["ldc"] + n
                C[c] = C[c] + v if pr["accumulate"] else v
    return C, rs


@pytest.mark.parametrize("trans_a,trans_b", [(0, 0), (0, 1), (1, 1), (1, 0)])
@pytest.mark.parametrize("epi", [(), ("bias", "relu"), ("bias", "relu", "rowdiv", "colscale"), ("mask", "res1", "res2"),
                                 ("bias", "rowdiv", "colscale", "mask", "res1", "rowsum")])
@pytest.mark.parametrize("accumulate", [0, 1])
def test_gemm_ref_matches_simt_epilogue_loop(trans_a, trans_b, epi, accumulate):
    """gemm_ref (the reference of the K3 kernel tests) against a plain loop over gemm_simt_kernel's epilogue order, two
    instances with their own slices of every operand, leading dimensions past N and K."""
    gen = torch.Generator().manual_seed(len(epi) * 8 + trans_a * 4 + trans_b * 2 + accumulate)
    pr = _gemm_problem(gen, 5, 6, 7, 2, trans_a, trans_b, accumulate, epi)
    out = R.gemm_ref(pr)
    C, rs = _gemm_loop(pr)
    assert rel(out["C"][0], C) < TOL
    written = out["C"][2]
    assert torch.equal(out["C"][0][~written], pr["C"][~written])          # nothing outside the instances' M x N blocks
    assert int(written.sum()) == 2 * 5 * 6
    assert bool((out["C"][1][written] > 0).all())
    if rs is not None:
        assert rel(out["rowsum"][0], rs) < TOL and int(out["rowsum"][2].sum()) == 2 * 5


def test_gemm_ref_bf16_rounds_operands_nearest_even():
    a = torch.tensor([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, 1.0 + 2.0 ** -9], dtype=torch.float64)
    assert R.bf16_round(a).tolist() == [1.0, 1.0 + 2.0 ** -6, 1.0]       # ties to even, below half down


def test_gemm_ref_gram_rows_follow_pack_indices():
    """With gram_z, row m of A is the packed upper triangle of G_m = Z_m^T Z_m in the slots of packing.pack_indices() (the
    16 padding slots zero), gram_f = ||G_m||_F + 1 and gram_g the rows, per instance at z * zs_gram_z."""
    from sgrl_b200.packing import GP_K, pack_indices
    gen = torch.Generator().manual_seed(5)
    M, N, nb, zs = 3, 4, 2, 3 * GP_K + 8
    Z = torch.randn(nb * zs, generator=gen, dtype=torch.float64)
    W = torch.randn(N * GP_K, generator=gen, dtype=torch.float64)
    pr = dict(M=M, N=N, K=GP_K, nb=nb, trans_a=0, trans_b=0, ldb=GP_K, ldc=N, zs_b=0, zs_c=M * N, alpha=1.0, accumulate=0,
              A=None, B=W, B_hi=None, C=torch.zeros(nb * M * N, dtype=torch.float64), gram_z=Z, zs_gram_z=zs,
              gram_f=torch.zeros(nb * zs, dtype=torch.float64), gram_g=torch.zeros(nb * zs, dtype=torch.float64))
    out = R.gemm_ref(pr)
    slots, ri, ci = pack_indices()
    for z in range(nb):
        for m in range(M):
            Zm = Z[z * zs + m * 96: z * zs + (m + 1) * 96].reshape(3, 32)
            G = Zm.T @ Zm
            row = torch.zeros(GP_K, dtype=torch.float64)
            for s, i, j in zip(slots, ri, ci):
                row[s] = G[i, j]
            assert rel(out["gram_g"][0][z * zs + m * GP_K: z * zs + (m + 1) * GP_K], row) < TOL
            assert abs(out["gram_f"][0][z * zs + m].item() - (G.norm().item() + 1.0)) < 1e-12 * G.norm().item()
            assert rel(out["C"][0][z * M * N + m * N: z * M * N + (m + 1) * N], W.reshape(N, GP_K) @ row) < TOL
    assert len(set(slots)) == 528
