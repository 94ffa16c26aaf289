"""fp64 references of the attention core (K2), the invariant features (K1) and the projections (K3) in the layouts of the C ABI
(include/sgrl_b200.h: sgrl_attention_fwd/bwd, sgrl_inv_feature_fwd/bwd, sgrl_gemm_desc).

Plain torch, no CUDA needed; every function computes in float64 on the device its inputs live on.  They restate
subequivariant_attentions.py:90-151 of the reference for packed variable-size graphs (token t = limb t - cu_limbs[g] of
graph g) and are pinned to the batched oracle (oracle/set_oracle.py) by tests/test_kernel_ref.py.  Graphs of equal size
are evaluated together (a gather of their token rows); nothing here depends on how the kernels walk the graphs.
"""
import torch

from sgrl_b200.packing import GP_K, pack_indices

HEADS, HD = 2, 128


def _graphs_by_size(cu_limbs):
    """{n: (graph indices (ng,), token indices (ng, n))} of the packed batch."""
    cu = cu_limbs.detach().to("cpu", torch.int64)
    t0, n = cu[:-1], cu[1:] - cu[:-1]
    out = {}
    for size in sorted(set(n.tolist())):
        g = torch.nonzero(n == size).flatten()
        out[size] = (g, t0[g][:, None] + torch.arange(size))
    return out


def _rel_tables(relation, rel_off, g, n):
    """(ng, n, n, 3) relation tables of graphs g: the one at rel_off[g] (0 when rel_off is None), indexed (i*n + j)*3."""
    off = torch.zeros(len(g), dtype=torch.int64) if rel_off is None else rel_off.detach().to("cpu", torch.int64)[g]
    idx = off[:, None] + torch.arange(n * n * 3)
    return relation.double()[idx.to(relation.device)].view(len(g), n, n, 3)


def _attention(qkv, vgp, gd, rel_w, rel_b, cu_limbs, rel_off, relation):
    """o (T,256), og (T,3,256), p (T,2,16) from fp64 tensors (differentiable in qkv, vgp, rel_w)."""
    T, dev = qkv.shape[0], qkv.device
    o = qkv.new_zeros(T, 2 * HD)
    og = qkv.new_zeros(T, 3, 2 * HD)
    p = qkv.new_zeros(T, HEADS, 16)
    for n, (g, tok) in _graphs_by_size(cu_limbs).items():
        ng, tok = len(g), tok.to(dev)
        x = qkv[tok]                                                        # (ng, n, 768)
        q, k, v = (x[..., c * 256:(c + 1) * 256].view(ng, n, HEADS, HD).transpose(1, 2) for c in range(3))
        S = q @ k.transpose(-1, -2)                                         # (ng, H, n, n)
        if rel_w is not None:
            rel = _rel_tables(relation, rel_off, g, n)
            S = S + torch.einsum("gijc,hc->ghij", rel, rel_w) + rel_b.view(1, HEADS, 1, 1)
        P = torch.softmax(S, dim=-1)                                        # over the graph's own limbs only
        o = o.index_put((tok.flatten(),), (P @ v).transpose(1, 2).reshape(ng * n, 2 * HD))
        # values of (r, h): [vgp[t, r*252 + h*126 : +126] | gd[t, r, 0:2]]
        vals = torch.cat([vgp[tok].view(ng, n, 3, HEADS, 126),
                          gd[tok].view(ng, n, 3, 1, 2).expand(ng, n, 3, HEADS, 2)], -1)
        og = og.index_put((tok.flatten(),), torch.einsum("ghij,gjrhc->girhc", P, vals).reshape(ng * n, 3, 2 * HD))
        p = p.index_put((tok.flatten(),), torch.nn.functional.pad(P.transpose(1, 2), (0, 16 - n)).reshape(ng * n, HEADS, 16))
    return o, og, p


def attention_fwd_ref(qkv, vgp, gd, rel_w, rel_b, cu_limbs, rel_off, relation):
    """sgrl_attention_fwd in fp64: qkv (T,768) = the stored (/F-divided, scaled) q|k|v, head h = columns h*128..h*128+127 of
    each; vgp (T,756) = (T,3,252); gd (T,6) = (T,3,2); rel_w (2,3), rel_b (2) or None; relation tables at rel_off[g]
    (None: all at 0).  Returns o (T,256), og (T,3,256), p (T,2,16) with p[t, h, j] = 0 for j >= n."""
    d = lambda t: None if t is None else t.detach().double()
    with torch.no_grad():
        return _attention(d(qkv), d(vgp).view(-1, 756), d(gd).view(-1, 6), d(rel_w), d(rel_b), cu_limbs, rel_off, relation)


def attention_bwd_ref(qkv, vgp, gd, rel_w, rel_b, cu_limbs, rel_off, relation, d_o, d_og):
    """sgrl_attention_bwd in fp64: the gradient of <d_o, o> + <d_og, og> w.r.t. the stored q|k|v (T,768), vgp (T,756) and
    rel_w (2,3) (None without a bias).  gd is an input of the network: no gradient."""
    x = qkv.detach().double().requires_grad_(True)
    vg = vgp.detach().double().reshape(-1, 756).requires_grad_(True)
    w = None if rel_w is None else rel_w.detach().double().requires_grad_(True)
    b = None if rel_b is None else rel_b.detach().double()
    with torch.enable_grad():
        o, og, _ = _attention(x, vg, gd.detach().double().view(-1, 6), w, b, cu_limbs, rel_off, relation)
        loss = (o * d_o.double().view(o.shape)).sum() + (og * d_og.double().view(og.shape)).sum()
        grads = torch.autograd.grad(loss, [x, vg] + ([w] if w is not None else []))
    return grads[0], grads[1], (grads[2] if w is not None else None)


def gram_packed(Z):
    """G = Z^T Z of Z (T,3,32) -> (G (T,32,32), packed upper triangle (T,544) in the slots of packing.pack_indices(), the
    16 padding slots 0)."""
    G = Z.transpose(-1, -2) @ Z
    slots, ri, ci = pack_indices()
    Gp = Z.new_zeros(Z.shape[0], GP_K)
    Gp[:, slots] = G[:, ri, ci]
    return G, Gp


def inv_feature_fwd_ref(X, v0, gd, P1, P2=None):
    """sgrl_inv_feature_fwd in fp64: X (T,3,128), v0 (T,3,8) or None (then C = 136, X = [v0 | X]), gd (T,3,2), P1, P2 (30,C).
    Z = [X P1^T | gd], Z2 = [X P2^T | gd] (None without P2), packed G of Z (T,544) and F = ||G||_F + 1 (T)."""
    with torch.no_grad():
        T = X.shape[0]
        x = X.double().reshape(T, 3, 128)
        if v0 is not None:
            x = torch.cat([v0.double().reshape(T, 3, 8), x], -1)
        g = gd.double().reshape(T, 3, 2)
        Z = torch.cat([x @ P1.double().t(), g], -1)
        Z2 = None if P2 is None else torch.cat([x @ P2.double().t(), g], -1)
        G, Gp = gram_packed(Z)
        F = torch.linalg.matrix_norm(G) + 1.0
    return Z, Z2, Gp, F


def inv_feature_bwd_ref(dGp, dF, Z):
    """sgrl_inv_feature_bwd in fp64: the gradient w.r.t. all 32 columns of Z (T,3,32) of
    sum_{i<=j} dGp[p(i,j)] G_ij + sum dF F.  This is the folded convention of the consumer GEMMs, dGp[p(i,j)] =
    dL/dG_ij + dL/dG_ji (i < j), dL/dG_ii on the diagonal; the padding slots of dGp do not enter."""
    slots, ri, ci = pack_indices()
    z = Z.detach().double().reshape(-1, 3, 32).requires_grad_(True)
    with torch.enable_grad():
        G = z.transpose(-1, -2) @ z
        F = torch.linalg.matrix_norm(G) + 1.0
        loss = (dGp.double().reshape(-1, GP_K)[:, slots] * G[:, ri, ci]).sum() + (dF.double().reshape(-1) * F).sum()
        (dz,) = torch.autograd.grad(loss, z)
    return dz


def bf16_round(x):
    """fp32 values rounded to bf16 with round-to-nearest-even (what the BF16-input mode feeds the tensor core), as fp64."""
    return x.float().to(torch.bfloat16).double()


def _mat(buf, off, rows, cols, ld, trans=False):
    """(rows, cols) matrix view of a flat buffer at element offset off: X[r][c] = buf[off + r*ld + c], or buf[off + c*ld + r]
    when trans."""
    return buf.as_strided((rows, cols), (1, ld) if trans else (ld, 1), off)


def gemm_ref(pr, bf16=False):
    """One SgrlGemmProblem of sgrl_gemm_desc in fp64.  pr: dict with the descriptor's fields, each pointer a flat tensor (or
    None) holding all nb instances at z * zs.  For every instance z:

        v = alpha * A B^T + bias -> relu -> / rowdiv -> * colscale (n < colscale_n) -> mask > 0 ? v : 0 -> + res1 + res2
        C = v, or C += v (accumulate);  columns 30, 31 of row m = 3t+r are gd[t][r][0..1] instead (gd)
        rowsum += alpha * sum_k A;  gram_z: row m of A = packed triangle of G_m = Z_m^T Z_m, gram_f = ||G_m||_F + 1, gram_g = rows

    (the order of gemm_simt_kernel's epilogue).  bf16: A and B rounded to bf16 (RN-even) before the product (B from B_hi when
    given: the kernel rounds the weights' hi part); rowsum sums the unrounded A.  Returns {name: (value, bound, written)}
    for C, rowsum, gram_f, gram_g: fp64 copies of the whole buffers with the computed entries replaced, a bound on each
    entry's magnitude built from the operands' absolute values (the scale of its rounding error) and the mask of the
    entries the call writes.  Everything else in a buffer must come back bit-identical."""
    M, N, K, nb = pr["M"], pr["N"], pr["K"], pr["nb"]
    d = {k: (v.detach().double().reshape(-1) if torch.is_tensor(v) else v) for k, v in pr.items()}
    out = {}
    for name in ("C", "rowsum", "gram_f", "gram_g"):
        if d.get(name) is not None:
            out[name] = (d[name].clone(), torch.zeros_like(d[name]), torch.zeros_like(d[name], dtype=torch.bool))
    Bsrc = d["B_hi"] if bf16 and d.get("B_hi") is not None else d["B"]
    alpha = float(pr.get("alpha", 1.0))
    with torch.no_grad():
        for z in range(nb):
            if d.get("gram_z") is not None:
                Z = _mat(d["gram_z"], z * d["zs_gram_z"], M, 96, 96).reshape(M, 3, 32)
                G, A = gram_packed(Z)
                F = (torch.linalg.matrix_norm(G) + 1.0)[:, None]
                for name, val, mag in (("gram_f", F, F), ("gram_g", A, gram_packed(Z.abs())[1])):
                    if name in out:
                        w = val.shape[1]
                        _mat(out[name][0], z * d["zs_gram_z"], M, w, w).copy_(val)
                        _mat(out[name][1], z * d["zs_gram_z"], M, w, w).copy_(mag)
                        _mat(out[name][2], z * d["zs_gram_z"], M, w, w).fill_(True)
            else:
                A = _mat(d["A"], z * d["zs_a"], M, K, d["lda"], bool(pr["trans_a"]))
            B = _mat(Bsrc, z * d["zs_b"], N, K, d["ldb"], bool(pr["trans_b"]))
            if "rowsum" in out:
                rs, rb, rw = out["rowsum"]
                o = z * d["zs_rowsum"]
                rb[o:o + M] = rs[o:o + M].abs() + abs(alpha) * A.abs().sum(1)
                rs[o:o + M] += alpha * A.sum(1)
                rw[o:o + M] = True
            Aq, Bq = (bf16_round(A), bf16_round(B)) if bf16 else (A, B)
            v = alpha * (Aq @ Bq.T)
            mag = abs(alpha) * (Aq.abs() @ Bq.abs().T)
            if d.get("bias") is not None:
                b = d["bias"][z * d["zs_bias"]: z * d["zs_bias"] + N]
                v = v + b
                mag = mag + b.abs()
            if pr.get("relu"):
                v = v.clamp_min(0.0)
            if d.get("rowdiv") is not None:
                r = d["rowdiv"][z * d["zs_rowdiv"]: z * d["zs_rowdiv"] + M, None]
                v = v / r
                mag = mag / r.abs()
            cn = min(int(pr.get("colscale_n", 0)), N)
            if cn > 0:
                cs = float(pr.get("colscale", 1.0))
                v[:, :cn] *= cs
                mag[:, :cn] *= abs(cs)
            if d.get("mask") is not None:
                v = torch.where(_mat(d["mask"], z * d["zs_mask"], M, N, d["ldmask"]) > 0, v, torch.zeros_like(v))
            for res, zs, ld in (("res1", "zs_res1", "ldres1"), ("res2", "zs_res2", "ldres2")):
                if d.get(res) is not None:
                    t = _mat(d[res], z * d[zs], M, N, d[ld])
                    v = v + t
                    mag = mag + t.abs()
            c, cb, cw = out["C"]
            dst = _mat(c, z * d["zs_c"], M, N, d["ldc"])
            if pr.get("accumulate"):
                mag = mag + dst.abs()
                v = dst + v
            if d.get("gd") is not None:
                gd = d["gd"][z * d["zs_gd"]: z * d["zs_gd"] + 2 * M].reshape(M, 2)
                v[:, 30:32] = gd if not pr.get("accumulate") else dst[:, 30:32] + gd
                mag[:, 30:32] = v[:, 30:32].abs()
            dst.copy_(v)
            _mat(cb, z * d["zs_c"], M, N, d["ldc"]).copy_(mag)
            _mat(cw, z * d["zs_c"], M, N, d["ldc"]).fill_(True)
    return out


# ======================================================================================================================
# The kernels around the projections (csrc/misc.cuh) and the triangle fold (csrc/feature.cuh), in the layouts of their entry
# points (sgrl_embed_fwd .. sgrl_unfold_sym) for ONE net instance: every operand a dense tensor of that net (the tests slice the
# instances out of their strided buffers).  Each takes the fp32 values the kernel reads and returns {output: (value, scale)} in
# float64, scale = the sum of the absolute values of the terms that form each element (the reference on absolute values where
# the map is linear; stated per kernel where it is not): the size of the rounding error an fp32 kernel can make there.
# ======================================================================================================================
S128 = 128.0 ** 0.5
LN_EPS = 1e-5


def _d(t):
    return None if t is None else t.detach().double()


def v0_of(obs):
    """V0 (T,3,8) with V0[r][j] = obs[3j + r] (SEActor.py:239-245)."""
    return obs[:, :24].reshape(-1, 8, 3).transpose(1, 2)


def pos_rows(E0, E1, E2, rank3):
    """ConcatPositionalEmbedding of each token: [E0[rank3[t,0]] | E1[rank3[t,1]] | E2[rank3[t,2]]] (T,128)."""
    r = rank3.long()
    return torch.cat([E0[r[:, 0]], E1[r[:, 1]], E2[r[:, 2]]], 1)


def embed_fwd_ref(obs, act, rank3, Wg, We, be, E0, E1, E2):
    """sgrl_embed_fwd: obs (T,41), act (T,3) for critics (We (128,20)) or None (We (128,17)).  V0 (T,24), GD (T,6), SH (T,ng),
    VG (T,3,128), H (T,128)."""
    obs, act, Wg, We, be = _d(obs), _d(act), _d(Wg), _d(We), _d(be)
    E0, E1, E2 = _d(E0), _d(E1), _d(E2)
    V0 = v0_of(obs)
    s0 = obs[:, 24:] if act is None else torch.cat([obs[:, 24:], act], 1)
    pos = pos_rows(E0, E1, E2, rank3)
    out = {"V0": (V0.reshape(-1, 24), None), "GD": (V0[:, :, 1:3].reshape(-1, 6), None), "SH": (s0, None),
           "VG": (S128 * V0 @ Wg.T, S128 * V0.abs() @ Wg.abs().T),
           "H": (S128 * (s0 @ We.T + be) + pos, S128 * (s0.abs() @ We.abs().T + be.abs()) + pos.abs())}
    return out


def _graph_gather(cu_limbs):
    """[(token indices (ng, n))] of the packed batch, one entry per graph size."""
    return [tok for _, (_, tok) in _graphs_by_size(cu_limbs).items()]


def _ingrad_loss(x, a, cu_limbs, L):
    """sum of <upstream, linear map of obs x> over every term input_grad_kernel gathers (csrc/misc.cuh), with the upstream
    gradients and coefficients in `a` (absolute values for the scale)."""
    V0 = v0_of(x)                                   # (T,3,8)
    s0 = x[:, 24:41]
    gd = V0[:, :, 1:3]                              # (T,3,2)
    loss = (a["dvg0"] * (S128 * V0 @ a["Wg"].T)).sum()                                 # Vg0 = sqrt(128) V0 Wg^T
    loss = loss + (a["dh0"] * (S128 * s0 @ a["We"][:, :17].T)).sum()                   # h0 = sqrt(128) We s0 (+ be + pos)
    for dz, W in ((a["dzh"], a["gg"]), (a["dzh2"], a["gph"])):                         # head invariants [V0 P[:, :8]^T | gd]
        if dz is not None:
            loss = loss + (dz[:, :, :30] * (V0 @ W[:, :8].T)).sum() + (dz[:, :, 30:32] * gd).sum()
    loss = loss + (a["dsh"][:, :17] * s0).sum()                                        # [s0 | h] -> linear1_ng
    for s in range(3 * L):                                                             # gd columns of every layer's Z1, Z2, Z3
        loss = loss + (a["dz"][s][:, :, 30:32] * gd).sum()
    for tok in _graph_gather(cu_limbs):                                                # gd in channels 126, 127 of the values
        tok = tok.to(x.device)
        n = tok.shape[1]
        g = gd[tok]                                                                    # (ng, n, 3, 2): key j
        for l in range(L):
            P = a["P"][l][tok][..., :n]                                                # (ng, n, 2, n): query i, head h, key j
            og = torch.einsum("gihj,gjrk->girhk", P, g)
            d = a["dog"][l][tok].view(*tok.shape, 3, 2, 128)[..., 126:128]             # (ng, n, 3, 2, 2)
            loss = loss + (d * og).sum()
    if a["dy"] is not None:                                                            # out_i = max_action tanh(sum_r V0[r][5+i] w_r)
        p = torch.einsum("tri,tr->ti", V0[:, :, 5:8], a["w3"])
        loss = loss + (a["dy"] * p).sum()
    return loss


def input_grad_ref(dvg0, dh0, dzh, dzh2, dsh, dz, dog, P, Wg, We, gg, gph, dout, out, w3, max_action, cu_limbs, L):
    """sgrl_input_grad for one net: d obs (T,41) = the gradient of _ingrad_loss.  dz: 3L tensors (T,3,32), dog: L (T,768),
    P: L (T,2,16); actor: dzh2 (T,3,32), gph (30,136), dout, out, w3 (T,3) (dy = dout max_action (1 - (out/max_action)^2), from
    the stored out as the kernel forms it), critic: all None.  Returns {"dobs": (value, scale)}."""
    T = dvg0.shape[0]
    a = {"dvg0": _d(dvg0).reshape(T, 3, 128), "dh0": _d(dh0).reshape(T, 128), "dzh": _d(dzh).reshape(T, 3, 32),
         "dzh2": None if dzh2 is None else _d(dzh2).reshape(T, 3, 32), "dsh": _d(dsh), "Wg": _d(Wg), "We": _d(We), "gg": _d(gg),
         "gph": _d(gph), "dz": [_d(t).reshape(T, 3, 32) for t in dz[:3 * L]], "dog": [_d(t).reshape(T, 768) for t in dog[:L]],
         "P": [_d(t).reshape(T, 2, 16) for t in P[:L]], "dy": None, "w3": _d(w3)}
    if dzh2 is not None:
        o = _d(out) / float(max_action)
        a["dy"] = _d(dout) * float(max_action) * (1.0 - o * o)
        a["dy_abs"] = _d(dout).abs() * float(max_action) * (1.0 + o * o)
    res = []
    for absval in (False, True):
        b = a
        if absval:
            b = {k: (None if v is None else [t.abs() for t in v] if isinstance(v, list) else v.abs()) for k, v in a.items()}
            if a["dy"] is not None:
                b["dy"] = a["dy_abs"]
        x = torch.zeros(T, 41, dtype=torch.float64, device=dvg0.device, requires_grad=True)
        with torch.enable_grad():
            (g,) = torch.autograd.grad(_ingrad_loss(x, b, cu_limbs, L), x)
        res.append(g)
    return {"dobs": tuple(res)}


def pos_embed_bwd_ref(dH, rank3):
    """sgrl_pos_embed_bwd: the gradients (15,42), (15,42), (15,44) of the three positional tables from dH (T,128)."""
    dH, r = _d(dH), rank3.long()
    out = {}
    for i, (c0, c1) in enumerate(((0, 42), (42, 84), (84, 128))):
        for name, src in (("v", dH), ("s", dH.abs())):
            t = torch.zeros(15, c1 - c0, dtype=torch.float64, device=dH.device).index_add_(0, r[:, i], src[:, c0:c1])
            out.setdefault(f"dE{i}", []).append(t)
    return {k: tuple(v) for k, v in out.items()}


def layernorm_fwd_ref(a, b, gamma, beta):
    """sgrl_layernorm_fwd: x = a + b (b None: x = a), y = (x - mean) rstd gamma + beta, rstd = (var + 1e-5)^-1/2, stats (T,2).
    Scales: x |a| + |b|; y |gamma| rstd (|x| + mean(|x|)) + |beta| (the rounding of x and of the mean, amplified by rstd); mean
    mean(|x|); rstd rstd (1 + mean(|x|) rstd) (the deviations' rounding relative to the standard deviation)."""
    a, b, g, be = _d(a), _d(b), _d(gamma), _d(beta)
    x = a if b is None else a + b
    xs = a.abs() if b is None else a.abs() + b.abs()
    mean = x.mean(1, keepdim=True)
    var = ((x - mean) ** 2).mean(1, keepdim=True)
    rstd = (var + LN_EPS).rsqrt()
    y = (x - mean) * rstd * g + be
    ax = x.abs().mean(1, keepdim=True)
    return {"x": (x, xs), "y": (y, g.abs() * rstd * (x.abs() + ax) + be.abs()),
            "mean": (mean[:, 0], ax[:, 0]), "rstd": (rstd[:, 0], (rstd * (1.0 + ax * rstd))[:, 0])}


def layernorm_bwd_ref(dy1, dy2, x, stats, gamma, rd_y=None, rd_F=None):
    """sgrl_layernorm_bwd from the stored stats (mean, rstd): with dy = dy1 + dy2 and xh = (x - mean) rstd,
    dx = rstd (g dy - mean(g dy) - xh mean(g dy xh)), dgamma = sum_t dy xh, dbeta = sum_t dy; the tail (rd_y, rd_F given):
    out = dx / F, dF = -<dx, y> / F.  Scales: the same expressions on absolute values."""
    dy = _d(dy1) if dy2 is None else _d(dy1) + _d(dy2)
    dys = _d(dy1).abs() if dy2 is None else _d(dy1).abs() + _d(dy2).abs()
    st, g = _d(stats), _d(gamma)
    mean, rstd = st[:, :1], st[:, 1:2]
    xh = (_d(x) - mean) * rstd
    gd = g * dy
    s1, s2 = gd.mean(1, keepdim=True), (gd * xh).mean(1, keepdim=True)
    dx = rstd * (gd - s1 - xh * s2)
    gds = g.abs() * dys
    dxs = rstd * (gds + gds.mean(1, keepdim=True) + xh.abs() * (gds * xh.abs()).mean(1, keepdim=True))
    out = {"dx": (dx, dxs), "dgamma": ((dy * xh).sum(0), (dys * xh.abs()).sum(0)), "dbeta": (dy.sum(0), dys.sum(0))}
    if rd_y is not None:
        F, y = _d(rd_F).reshape(-1, 1), _d(rd_y)
        out["rd_out"] = (dx / F, dxs / F.abs())
        out["rd_dF"] = (-(dx * y).sum(1) / F[:, 0], (dxs * y.abs()).sum(1) / F[:, 0].abs())
    return out


def matapply_fwd_ref(Z, M):
    """sgrl_matapply_fwd: R = Z (3x32) M (32x32) per token; Z (T,3,32), M (T,32,32)."""
    Z, M = _d(Z).reshape(-1, 3, 32), _d(M).reshape(-1, 32, 32)
    return {"R": (Z @ M, Z.abs() @ M.abs())}


def _matapply_bwd(dR, dRs, Z, M, F):
    dM, dMs = Z.transpose(1, 2) @ dR, Z.abs().transpose(1, 2) @ dRs
    F = F.reshape(-1, 1, 1)
    return {"dZ": (dR @ M.transpose(1, 2), dRs @ M.abs().transpose(1, 2)), "dT": (dM / F, dMs / F.abs()),
            "dF": (-(dM * M).sum((1, 2)) / F[:, 0, 0], (dMs * M.abs()).sum((1, 2)) / F[:, 0, 0].abs())}


def matapply_bwd_ref(dR, Z, M, F):
    """sgrl_matapply_bwd with M = Tm / F: dZ = dR M^T, dT = Z^T dR / F, dF = -<Z^T dR, M> / F."""
    dR = _d(dR).reshape(-1, 3, 32)
    return _matapply_bwd(dR, dR.abs(), _d(Z).reshape(-1, 3, 32), _d(M).reshape(-1, 32, 32), _d(F))


def matapply_l5_fwd_ref(Z, M, W5, Vg, dV):
    """sgrl_matapply_l5_fwd: R = Z M, Vn = Vg + dV + R W5^T; W5 (128,32), Vg, dV (T,3,128)."""
    r = matapply_fwd_ref(Z, M)["R"]
    W5, Vg, dV = _d(W5), _d(Vg).reshape(-1, 3, 128), _d(dV).reshape(-1, 3, 128)
    return {"R": r, "Vn": (Vg + dV + r[0] @ W5.T, Vg.abs() + dV.abs() + r[1] @ W5.abs().T)}


def matapply_l5_bwd_ref(dVn, W5, Z, M, F):
    """sgrl_matapply_l5_bwd: dR = dVn W5, then matapply_bwd_ref's math."""
    dVn, W5 = _d(dVn).reshape(-1, 3, 128), _d(W5)
    return _matapply_bwd(dVn @ W5, dVn.abs() @ W5.abs(), _d(Z).reshape(-1, 3, 32), _d(M).reshape(-1, 32, 32), _d(F))


def actor_out_fwd_ref(R, V0, wd, max_action):
    """sgrl_actor_out_fwd: w_r = sum_c R[r][c] wd[c] (W3), p_i = sum_r V0[r][5+i] w_r, out = max_action tanh(p).  Scale of out:
    max_action ((1 - tanh^2) scale(p) + |tanh p|) (the argument's rounding through the slope, and tanhf's own)."""
    R, V0, wd = _d(R).reshape(-1, 3, 32), _d(V0).reshape(-1, 3, 8), _d(wd).reshape(32)
    w, ws = R @ wd, R.abs() @ wd.abs()
    ax = V0[:, :, 5:8]
    p = torch.einsum("tri,tr->ti", ax, w)
    ps = torch.einsum("tri,tr->ti", ax.abs(), ws)
    a = torch.tanh(p)
    return {"W3": (w, ws), "out": (max_action * a, max_action * ((1 - a * a) * ps + a.abs())), "p": (p, ps)}


def actor_out_bwd_ref(dout, out, R, V0, wd, max_action):
    """sgrl_actor_out_bwd from the stored out: a = out / max_action, dp = dout max_action (1 - a^2), dw_r = sum_i dp_i V0[r][5+i],
    dR = dw wd^T, dwd = sum_t sum_r dw_r R[r]."""
    a = _d(out) / float(max_action)
    do = _d(dout)
    dp, dps = do * float(max_action) * (1 - a * a), do.abs() * float(max_action) * (1 + a * a)
    R, V0, wd = _d(R).reshape(-1, 3, 32), _d(V0).reshape(-1, 3, 8), _d(wd).reshape(32)
    ax = V0[:, :, 5:8]
    dw, dws = torch.einsum("tri,ti->tr", ax, dp), torch.einsum("tri,ti->tr", ax.abs(), dps)
    return {"dR": (dw[..., None] * wd, dws[..., None] * wd.abs()),
            "dwd": ((dw[..., None] * R).sum((0, 1)), (dws[..., None] * R.abs()).sum((0, 1)))}


def rowdiv_bwd_ref(g, y, F, colscale, cs_n):
    """sgrl_rowdiv_bwd: with y = t / F (* colscale on columns < cs_n) and upstream g (T,N): dt = g cs / F, dF = -<g, y> / F."""
    g, y, F = _d(g), _d(y), _d(F).reshape(-1, 1)
    cs = torch.ones(g.shape[1], dtype=torch.float64, device=g.device)
    cs[:cs_n] = float(colscale)
    return {"dt": (g * cs / F, g.abs() * cs.abs() / F.abs()),
            "dF": (-(g * y).sum(1) / F[:, 0], (g.abs() * y.abs()).sum(1) / F[:, 0].abs())}


def colsum_ref(X, alpha):
    """sgrl_colsum: alpha * sum_m X[m][n] (added to the output)."""
    X = _d(X)
    return {"out": (float(alpha) * X.sum(0), abs(float(alpha)) * X.abs().sum(0))}


def fold_ref(W):
    """sgrl_fold_sym of one (rows,1024) weight in fp32, as the kernel adds: W'[o][p(i,j)] = W[o][32i+j] + W[o][32j+i] (i < j),
    W[o][33i] (i = j), in the slots of packing.pack_indices(); the 16 padding slots 0."""
    slots, ri, ci = pack_indices()
    ri, ci = torch.tensor(ri, device=W.device), torch.tensor(ci, device=W.device)
    Wf = W.new_zeros(W.shape[0], GP_K)
    Wf[:, slots] = torch.where(ri == ci, W[:, ri * 32 + ci], W[:, ri * 32 + ci] + W[:, ci * 32 + ri])
    return Wf


def unfold_ref(gf):
    """sgrl_unfold_sym's term for one (rows,544) folded gradient: dW[o][32a+b] = gf[o][p(min(a,b), max(a,b))] (rows,1024)."""
    slots, ri, ci = pack_indices()
    dW = gf.new_zeros(gf.shape[0], 32, 32)
    ri, ci, sl = (torch.tensor(v, device=gf.device) for v in (ri, ci, slots))
    dW[:, ri, ci] = gf[:, sl]
    dW[:, ci, ri] = gf[:, sl]
    return dW.reshape(-1, 1024)
