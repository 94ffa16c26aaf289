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


# ---- the kernels around the projections (csrc/misc.cuh) and the triangle fold -------------------------------------------------
def _embed_inputs(name, B, kind):
    """Oracle parameters (fp64), the network input x (B,N,41|44), the graph and the packed per-token operands of the embedding."""
    par = M.ALL[name]
    N = len(par)
    g = G.build_graph(par)
    p = {k: v.double() for k, v in O.synth_params(kind, 5).items()}
    b = synth.make_batch(B, N, seed=4)
    obs = b["obs"].view(B * N, 41).double()
    act = b["action"].view(B * N, 3).double() if kind == "critic" else None
    rank3 = torch.stack(g["traversals"], 1).repeat(B, 1).int()                 # (T,3): token t = limb t % N
    return p, g, obs, act, rank3, N


@pytest.mark.parametrize("name,B", CASES)
@pytest.mark.parametrize("kind", ["actor", "critic"])
def test_embed_fwd_ref_reproduces_oracle(name, B, kind):
    """embed_fwd_ref's V0, GD, SH, VG and H against the input stage of transformer_model (trace V0, GD, SH, 0.VGIN) and
    pos_embedding: h0 = (We s0 + be) sqrt(128) + pos."""
    p, g, obs, act, rank3, N = _embed_inputs(name, B, kind)
    T = B * N
    x = obs.view(B, N, 41) if act is None else torch.cat([obs.view(B, N, 41), act.view(B, N, 3)], 2)
    tr = {}
    with torch.no_grad():
        O.transformer_model(p, x, dict(g, relation=g["relation"].double()), trace=tr)
    E = [p[f"pos_encoder.embeddings.{i}.weight"] for i in range(3)]
    r = R.embed_fwd_ref(obs, act, rank3, p["g_encoder.weight"], p["encoder.weight"], p["encoder.bias"], *E)
    assert rel(r["V0"][0], _tok(tr["V0"], T)) < TOL and rel(r["GD"][0], _tok(tr["GD"], T)) < TOL
    ng = 17 if kind == "actor" else 20
    assert rel(r["SH"][0], _tok(tr["SH"], T)[:, :ng]) < TOL
    assert rel(r["VG"][0].reshape(T, -1), _tok(tr["0.VGIN"], T)) < TOL
    s0 = x.reshape(T, -1)[:, 24:]
    h0 = (s0 @ p["encoder.weight"].T + p["encoder.bias"]) * 128 ** 0.5 + O.pos_embedding(p, g["traversals"]).repeat(B, 1)
    assert rel(r["H"][0], h0) < TOL
    for k in ("VG", "H"):
        assert bool((r[k][1] >= r[k][0].abs()).all())


@pytest.mark.parametrize("a_mean,a_std", [(0.0, 1.0), (1e3, 1e-2), (5.0, 0.0)])
@pytest.mark.parametrize("resid", [False, True])
def test_layernorm_fwd_ref_matches_torch(a_mean, a_std, resid):
    gen = torch.Generator().manual_seed(int(a_mean) + resid)
    T = 6
    a = a_mean + a_std * torch.randn(T, 128, generator=gen, dtype=torch.float64)
    b = 0.1 * a_std * torch.randn(T, 128, generator=gen, dtype=torch.float64) if resid else None
    gamma, beta = torch.randn(128, generator=gen, dtype=torch.float64), torch.randn(128, generator=gen, dtype=torch.float64)
    r = R.layernorm_fwd_ref(a, b, gamma, beta)
    x = a if b is None else a + b
    y = torch.nn.functional.layer_norm(x, (128,), gamma, beta, eps=1e-5)
    assert bool(((r["y"][0] - y).abs() <= 1e-13 * r["y"][1]).all())        # torch's fp64 rounding, within the stated scale
    assert rel(r["x"][0], x) < TOL
    assert rel(r["mean"][0], x.mean(1)) < TOL
    assert bool(((r["rstd"][0] - 1 / (x.var(1, unbiased=False) + 1e-5).sqrt()).abs() <= 1e-13 * r["rstd"][1]).all())


@pytest.mark.parametrize("tail", [False, True])
@pytest.mark.parametrize("second", [False, True])
def test_layernorm_bwd_ref_matches_autograd(tail, second):
    """dx, dgamma, dbeta against autograd of <dy1 + dy2, LN(a + f)>; with the tail f = t / F also d t (rd_out) and d F (rd_dF)."""
    gen = torch.Generator().manual_seed(tail * 2 + second)
    T = 5
    a = torch.randn(T, 128, generator=gen, dtype=torch.float64)
    t = torch.randn(T, 128, generator=gen, dtype=torch.float64).requires_grad_(True)
    Fn = (torch.rand(T, generator=gen, dtype=torch.float64) * 3 + 0.5).requires_grad_(True)
    gamma = torch.randn(128, generator=gen, dtype=torch.float64).requires_grad_(True)
    beta = torch.randn(128, generator=gen, dtype=torch.float64).requires_grad_(True)
    dy1 = torch.randn(T, 128, generator=gen, dtype=torch.float64)
    dy2 = torch.randn(T, 128, generator=gen, dtype=torch.float64) if second else None
    ain = a.clone().requires_grad_(True)
    f = t / Fn[:, None]
    x = ain + f if tail else ain
    y = torch.nn.functional.layer_norm(x, (128,), gamma, beta, eps=1e-5)
    dy = dy1 if dy2 is None else dy1 + dy2
    (y * dy).sum().backward()
    fw = R.layernorm_fwd_ref(x.detach(), None, gamma.detach(), beta.detach())
    stats = torch.stack([fw["mean"][0], fw["rstd"][0]], 1)
    r = R.layernorm_bwd_ref(dy1, dy2, x.detach(), stats, gamma, f.detach() if tail else None, Fn.detach() if tail else None)
    assert rel(r["dx"][0], ain.grad) < 1e-12
    assert rel(r["dgamma"][0], gamma.grad) < 1e-12 and rel(r["dbeta"][0], beta.grad) < 1e-12
    if tail:
        assert rel(r["rd_out"][0], t.grad) < 1e-12 and rel(r["rd_dF"][0], Fn.grad) < 1e-12


def test_matapply_refs_match_autograd():
    """matapply_bwd_ref with M = Tm / F and matapply_l5_bwd_ref (dR = dVn W5) against autograd of the forward references."""
    gen = torch.Generator().manual_seed(11)
    T = 4
    Z = torch.randn(T, 3, 32, generator=gen, dtype=torch.float64).requires_grad_(True)
    Tm = torch.randn(T, 32, 32, generator=gen, dtype=torch.float64).requires_grad_(True)
    Fn = (torch.rand(T, generator=gen, dtype=torch.float64) * 2 + 0.1).requires_grad_(True)
    W5 = torch.randn(128, 32, generator=gen, dtype=torch.float64).requires_grad_(True)
    Vg, dV = torch.randn(T, 3, 128, generator=gen, dtype=torch.float64), torch.randn(T, 3, 128, generator=gen, dtype=torch.float64)
    Mm = Tm / Fn[:, None, None]
    dR = torch.randn(T, 3, 32, generator=gen, dtype=torch.float64)
    R0 = Z @ Mm
    assert rel(R.matapply_fwd_ref(Z, Mm)["R"][0], R0) < TOL
    (R0 * dR).sum().backward()
    r = R.matapply_bwd_ref(dR, Z, Mm.detach(), Fn)
    assert rel(r["dZ"][0], Z.grad) < 1e-12 and rel(r["dT"][0], Tm.grad) < 1e-12 and rel(r["dF"][0], Fn.grad) < 1e-12
    Z.grad = Tm.grad = Fn.grad = None
    Mm = Tm / Fn[:, None, None]
    f5 = R.matapply_l5_fwd_ref(Z, Mm, W5, Vg, dV)
    Vn = Vg + dV + (Z @ Mm) @ W5.T
    assert rel(f5["Vn"][0], Vn) < TOL and rel(f5["R"][0], Z @ Mm) < TOL
    dVn = torch.randn(T, 3, 128, generator=gen, dtype=torch.float64)
    (Vn * dVn).sum().backward()
    r = R.matapply_l5_bwd_ref(dVn, W5, Z, Mm.detach(), Fn)
    assert rel(r["dZ"][0], Z.grad) < 1e-12 and rel(r["dT"][0], Tm.grad) < 1e-12 and rel(r["dF"][0], Fn.grad) < 1e-12


@pytest.mark.parametrize("max_action", [0.4, 2.5])
def test_actor_out_refs_match_oracle_and_autograd(max_action):
    """actor_out_fwd_ref against the oracle's actor head (transformer_model's output axes . w, then SEPolicy's tanh), and
    actor_out_bwd_ref (from the stored out) against autograd of <dout, out> w.r.t. R and wd."""
    gen = torch.Generator().manual_seed(int(max_action * 10))
    T = 6
    Rh = torch.randn(T, 3, 32, generator=gen, dtype=torch.float64).requires_grad_(True)
    V0 = torch.randn(T, 3, 8, generator=gen, dtype=torch.float64)
    wd = torch.randn(1, 32, generator=gen, dtype=torch.float64).requires_grad_(True)
    w = torch.nn.functional.linear(Rh, wd).squeeze(-1)                         # set_oracle.transformer_model :275-285
    out = max_action * torch.tanh(torch.einsum("bri,br->bi", V0[..., 5:8], w))
    f = R.actor_out_fwd_ref(Rh, V0, wd, max_action)
    assert rel(f["out"][0], out) < TOL and rel(f["W3"][0], w) < TOL
    dout = torch.randn(T, 3, generator=gen, dtype=torch.float64)
    (out * dout).sum().backward()
    b = R.actor_out_bwd_ref(dout, out.detach(), Rh, V0, wd, max_action)
    assert rel(b["dR"][0], Rh.grad) < 1e-12 and rel(b["dwd"][0], wd.grad[0]) < 1e-12


def test_rowdiv_and_pos_embed_bwd_refs_match_autograd():
    gen = torch.Generator().manual_seed(3)
    T, N = 5, 40
    t = torch.randn(T, N, generator=gen, dtype=torch.float64).requires_grad_(True)
    Fn = (torch.rand(T, generator=gen, dtype=torch.float64) * 5 + 0.05).requires_grad_(True)
    cs = torch.ones(N, dtype=torch.float64)
    cs[:7] = 0.3
    y = t / Fn[:, None] * cs
    g = torch.randn(T, N, generator=gen, dtype=torch.float64)
    (y * g).sum().backward()
    r = R.rowdiv_bwd_ref(g, y.detach(), Fn, 0.3, 7)
    assert rel(r["dt"][0], t.grad) < 1e-12 and rel(r["dF"][0], Fn.grad) < 1e-12

    par = M.ALL["3d_humanoid_9_full"]
    gr = G.build_graph(par)
    p = {k: v.double().requires_grad_(True) for k, v in O.synth_params("actor", 2).items() if k.startswith("pos_encoder")}
    B = 3
    pos = O.pos_embedding(p, gr["traversals"]).repeat(B, 1)
    dH = torch.randn(B * len(par), 128, generator=gen, dtype=torch.float64)
    (pos * dH).sum().backward()
    r = R.pos_embed_bwd_ref(dH, torch.stack(gr["traversals"], 1).repeat(B, 1))
    for i in range(3):
        assert rel(r[f"dE{i}"][0], p[f"pos_encoder.embeddings.{i}.weight"].grad) < 1e-12
    assert rel(R.colsum_ref(dH, -0.5)["out"][0], -0.5 * dH.sum(0)) < TOL


@pytest.mark.parametrize("actor", [True, False])
def test_input_grad_ref_matches_per_token_formulas(actor):
    """input_grad_ref (autograd of the summed linear terms) against the per-token formulas of input_grad_kernel's comment
    (csrc/misc.cuh) written out element by element, on ragged graphs of 2, 5 and 16 limbs and L = 2."""
    gen = torch.Generator().manual_seed(int(actor))
    sizes, L, ng, ma = [2, 5, 16], 2, (17 if actor else 20), 2.5
    cu = torch.tensor([0] + list(torch.tensor(sizes).cumsum(0)), dtype=torch.int32)
    T = int(cu[-1])
    rn = lambda *s: torch.randn(*s, generator=gen, dtype=torch.float64)
    dvg0, dh0, dzh, dsh = rn(T, 3, 128), rn(T, 128), rn(T, 3, 32), rn(T, ng + 128)
    dzh2 = rn(T, 3, 32) if actor else None
    dz = [rn(T, 3, 32) for _ in range(3 * L)]
    dog = [rn(T, 768) for _ in range(L)]
    P = [rn(T, 2, 16).abs() for _ in range(L)]
    Wg, We, gg = rn(128, 8), rn(128, ng), rn(30, 136)
    gph = rn(30, 136) if actor else None
    dout, w3 = rn(T, 3), rn(T, 3)
    out = ma * torch.tanh(rn(T, 3))
    got = R.input_grad_ref(dvg0, dh0, dzh, dzh2, dsh, dz, dog, P, Wg, We, gg, gph, dout if actor else None,
                           out if actor else None, w3, ma, cu, L)["dobs"][0]
    s = 128 ** 0.5
    want = torch.zeros(T, 41, dtype=torch.float64)
    for t in range(T):
        g = int(torch.searchsorted(cu, torch.tensor(t, dtype=torch.int32), right=True)) - 1
        t0, n = int(cu[g]), int(cu[g + 1] - cu[g])
        dV0 = s * dvg0[t] @ Wg                                             # (3,8)
        for dzx, W in ((dzh, gg), (dzh2, gph)):
            if dzx is not None:
                dV0 += dzx[t, :, :30] @ W[:, :8]
                dV0[:, 1:3] += dzx[t, :, 30:32]
        for d in dz:
            dV0[:, 1:3] += d[t, :, 30:32]
        for l in range(L):
            for i in range(n):
                for h in range(2):
                    dV0[:, 1:3] += P[l][t0 + i, h, t - t0] * dog[l][t0 + i].view(3, 2, 128)[:, h, 126:128]
        if actor:
            a = out[t] / ma
            dy = dout[t] * ma * (1 - a * a)
            dV0[:, 5:8] += w3[t][:, None] * dy[None, :]
        for r in range(3):
            for j in range(8):
                want[t, 3 * j + r] = dV0[r, j]
        want[t, 24:] = s * dh0[t] @ We[:, :17] + dsh[t, :17]
    assert rel(got, want) < 1e-12


def test_fold_and_unfold_refs_follow_pack_indices():
    """fold_ref's W' contracts the packed triangle of a symmetric G like vec(G) contracts W, and unfold_ref of dW' is the gradient
    of that contraction w.r.t. W (the algebra of tests/test_fold_math.py, in the layout of sgrl_fold_sym / sgrl_unfold_sym)."""
    from sgrl_b200.packing import pack_indices
    gen = torch.Generator().manual_seed(9)
    slots, ri, ci = pack_indices()
    W = torch.randn(5, 1024, generator=gen, dtype=torch.float64).requires_grad_(True)
    Z = torch.randn(4, 3, 32, generator=gen, dtype=torch.float64)
    Gf, Gp = R.gram_packed(Z)
    Wf = R.fold_ref(W.detach())
    pad = sorted(set(range(544)) - set(slots))
    assert torch.all(Wf[:, pad] == 0)
    y = Gf.reshape(4, 1024) @ W.T
    assert rel(Gp @ Wf.T, y.detach()) < 1e-13
    dy = torch.randn(4, 5, generator=gen, dtype=torch.float64)
    (y * dy).sum().backward()
    assert rel(R.unfold_ref(dy.T @ Gp), W.grad) < 1e-13
