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
