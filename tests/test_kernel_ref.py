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
