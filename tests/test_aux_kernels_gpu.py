"""The kernels around the projections (csrc/misc.cuh) and the triangle fold (csrc/feature.cuh) checked directly against fp64
(tests/kernel_ref.py) through their single-kernel entry points (include/sgrl_b200.h, sgrl_embed_fwd .. sgrl_unfold_sym), which
launch through the same host launchers as the network passes, in every launch regime the update and the rollout reach:

  one token per warp (grid_for_warps: 8 x 148 CTAs of 8 warps), warps walking tokens above 9 472 tokens
      layernorm_fwd, rowdiv_bwd, matapply_fwd / _bwd, matapply_l5_fwd / _bwd, actor_out_fwd
  296 CTAs, warps walking tokens above 2 368, per-CTA partial weight gradients combined by atomics; one CTA in deterministic mode
      layernorm_bwd (+ dgamma, dbeta), actor_out_bwd (+ dwd), input_grad (no atomics)
  592 CTAs of 8-token groups walking above 4 736 tokens, a partial last group when T % 8 != 0      embed_fwd
  ceil(T / 64) CTAs of contiguous token ranges, at most 148; one CTA in deterministic mode         pos_embed_bwd
  y-split min(ceil(M / 64), 32) of the rows; one slice in deterministic mode                       colsum
  at most 592 CTAs walking the elements                                                             block_copy

Every case
  - gives every net instance z its own slice of every operand at z * zs, with zs past the dense size (the gap is NaN: a wrong
    z-stride reads NaN or writes where nothing may be written), and NaN in every output element the call does not write,
    pad rows past T and pad columns of strided outputs included: they must come back bit-identical;
  - starts every accumulating output (dF, dgamma, dbeta, dwd, the positional-table gradients, colsum's output, the unfolded
    gradients) from random values and compares it with prefill + reference;
  - bounds each element's error by its own scale (kernel_ref: the sum of the absolute values of the terms that form it; stated
    per kernel for the LayerNorms and the tanh) and reports the worst element as (z, t, column);
  - asserts the grid the entry point reports, and test_regime_coverage pins the (kernel, regime) pairs the cases reach.
block_copy, fold_sym (and its tf32 hi / lo planes), unfold_sym and the V0 / GD / SH copies of embed_fwd are checked bit for bit.

Tolerances: 4x the worst ratio measured on a B200 (power limit 1000 W), see TOL.
"""
import ctypes as C
import math

import pytest
import torch

import kernel_ref as R
from sgrl_b200.packing import GP_K, pack_indices

pytestmark = pytest.mark.gpu

NAN = float("nan")
WARP_CAP, BWD_CAP, EMBED_CAP = 8 * 148, 2 * 148, 4 * 148          # CTAs
TOL = {       # 4x the worst ratio measured on a B200 at a 1000 W power limit (in the comments; the worse of two runs), rounded up
    "embed_fwd.VG": 1.2e-6, "embed_fwd.H": 1.5e-6,                                   # 2.9e-7, 3.5e-7
    "input_grad.dobs": 3.7e-7,                                                        # 9.1e-8
    "pos_embed_bwd.dE": 7.6e-7,                                                       # 1.9e-7
    "layernorm_fwd.x": 2.4e-7, "layernorm_fwd.y": 8.6e-7, "layernorm_fwd.stats": 6.6e-7,    # 6.0e-8, 2.1e-7, 1.6e-7
    "layernorm_bwd.dx": 6.9e-7, "layernorm_bwd.dgamma": 5.4e-7,                       # 1.7e-7, 1.3e-7 (dgamma and dbeta)
    "layernorm_bwd.rd_out": 7.9e-7, "layernorm_bwd.rd_dF": 1.4e-7,                    # 2.0e-7, 3.4e-8
    "matapply_fwd.R": 1.6e-6,                                                         # 3.9e-7
    "matapply_bwd.dZ": 1.4e-6, "matapply_bwd.dT": 1e-6, "matapply_bwd.dF": 1.8e-7,    # 3.3e-7, 2.5e-7, 4.4e-8
    "matapply_l5_fwd.R": 1.4e-6, "matapply_l5_fwd.Vn": 4.2e-7,                        # 3.4e-7, 1.0e-7
    "matapply_l5_bwd.dZ": 2.6e-7, "matapply_l5_bwd.dT": 1.6e-6, "matapply_l5_bwd.dF": 3.6e-8,   # 6.3e-8, 3.8e-7, 9.0e-9
    "actor_out_fwd.W3": 4.9e-7, "actor_out_fwd.out": 3.1e-7,                         # 1.2e-7, 7.7e-8
    "actor_out_bwd.dR": 8.6e-7, "actor_out_bwd.dwd": 6.3e-9,                          # 2.1e-7, 1.6e-9
    "rowdiv_bwd.dt": 7e-7, "rowdiv_bwd.dF": 6.9e-7,                                   # 1.7e-7, 1.7e-7
    "colsum.out": 1.4e-7,                                                             # 3.4e-8
}


def r4(n):
    return (n + 3) // 4 * 4


class Buf:
    """nb instances of a per-net buffer of `dense` floats: instance z at z * zs, zs = dense plus a gap, 64 floats past the
    last instance; NaN wherever nothing is filled in."""

    def __init__(self, nb, dense):
        self.nb, self.zs = nb, r4(dense) + r4(dense // 3) + 20
        self.t = torch.full((nb * self.zs + 64,), NAN, device="cuda")

    def view(self, z, rows, cols, ld, off=0):
        return self.t.as_strided((rows, cols), (ld, 1), z * self.zs + off)

    def ptr(self, off=0):
        return self.t.data_ptr() + self.t.element_size() * off


class Layout:
    """Operands of one arena (stash, workspace, parameters, gradients) of nb nets: add(name, rows, ld) reserves a (rows, ld)
    region at a 16-byte aligned offset off[name], followed by 4 unused floats; build() allocates."""

    def __init__(self):
        self.n, self.off = 0, {}

    def add(self, name, rows, ld):
        self.off[name] = self.n
        self.n = r4(self.n + rows * ld + 4)

    def build(self, nb):
        return Buf(nb, self.n)


def rnd(gen, rows, cols, scale=1.0, shift=0.0):
    return torch.randn(rows, cols, device="cuda", generator=gen) * scale + shift


class Want:
    """What a buffer must hold after the call: the expected value and scale of every element it writes, bit-identical
    elsewhere."""

    def __init__(self, buf):
        self.buf = buf
        self.before = buf.t.clone()
        self.val = self.before.double()
        self.scale = torch.zeros_like(self.val)
        self.mask = torch.zeros_like(self.val, dtype=torch.bool)
        self.where = {}

    def set(self, z, rows, cols, ld, off, val, scale=None, acc=False):
        """expected val (fp64) with scale (None: bit for bit); acc: the region held random prefill that the call adds to."""
        o = z * self.buf.zs + off
        v = self.val.as_strided((rows, cols), (ld, 1), o)
        s = self.scale.as_strided((rows, cols), (ld, 1), o)
        val = val.reshape(rows, cols).double()
        if acc:
            s.copy_(v.abs() + (0 if scale is None else scale.reshape(rows, cols)))
            v.copy_(v + val)
        else:
            v.copy_(val)
            s.copy_(0 if scale is None else scale.reshape(rows, cols))
        self.mask.as_strided((rows, cols), (ld, 1), o).fill_(True)
        self.where[o] = (z, ld)

    def measure(self, label):
        """(worst ratio |got - want| / scale, where); asserts the sentinels and that every written element is finite."""
        got = self.buf.t
        keep = ~self.mask
        changed = got.view(torch.int32)[keep] != self.before.view(torch.int32)[keep]
        if changed.any():
            i = int(torch.nonzero(keep)[int(torch.nonzero(changed)[0])])
            raise AssertionError(f"{label}: element {self.loc(i)} outside the written region changed: {got[i].item()!r}")
        idx = torch.nonzero(self.mask).flatten()
        g = got.double()[idx]
        assert torch.isfinite(g).all(), f"{label}: non-finite value at {self.loc(int(idx[int(torch.nonzero(~torch.isfinite(g))[0])]))}"
        return self.worst(self.mask)

    def worst(self, mask):
        """worst |got - want| / scale over the elements of mask, and where (None, None when the mask is empty)"""
        idx = torch.nonzero(mask).flatten()
        if idx.numel() == 0:
            return None, None
        g = self.buf.t.double()[idx]
        d = (g - self.val[idx]).abs()
        ratio = torch.where(d == 0, torch.zeros_like(d), d / self.scale[idx])
        i = int(ratio.argmax())
        return ratio[i].item(), f"{self.loc(int(idx[i]))}: {g[i].item():.9g} vs {self.val[idx[i]].item():.9g}"

    def loc(self, i):
        o = max((o for o in self.where if o <= i), default=None)
        if o is None:
            return f"flat {i}"
        z, ld = self.where[o]
        return f"(z={z}, t={(i - o) // ld}, col={(i - o) % ld})"


class Run:
    """What one case reached: the grids and regimes, and the worst ratio per checked output."""

    def __init__(self):
        self.regimes, self.ratios = set(), []

    def grid(self, kernel, regime, got, want):
        assert tuple(got) == tuple(want), f"{kernel}: launched grid {tuple(got)}, expected {tuple(want)} ({regime})"
        self.regimes.add((kernel, regime))

    def check(self, label, want):
        w, where = want.measure(label)
        self.ratios.append((label, w, where))


def lib():
    from sgrl_b200._lib import lib as L
    return L


def call(name, *args):
    from sgrl_b200._lib import check, stream
    grid = (C.c_int32 * 3)()
    check(getattr(lib(), name)(*args, grid, stream()), name)
    torch.cuda.synchronize()
    return list(grid)


def det(on):
    return lib().sgrl_deterministic(1 if on else 0)


def warp_grid(T, cap=WARP_CAP):
    return min(max((T + 7) // 8, 1), cap)


def warp_regime(T, cap=WARP_CAP):
    return "walk" if (T + 7) // 8 > cap else "warp-per-token"


def f_divisors(gen, T):
    """F (T) spread log-uniformly over 0.05 .. 50."""
    return torch.exp(torch.rand(T, device="cuda", generator=gen) * math.log(1000.0) + math.log(0.05))


# ================================================================================================================= embed_fwd
def embed_case(r, T, nb, in_nets, kind, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    ng = 17 if kind == "actor" else 20
    KS = 128 + ng
    obs = Buf(in_nets, 41 * T)
    act = Buf(in_nets, 3 * T) if kind == "critic" else None
    for b in range(in_nets):
        obs.view(b, T, 41, 41).copy_(rnd(gen, T, 41))
        if act:
            act.view(b, T, 3, 3).copy_(rnd(gen, T, 3))
    rank3 = torch.randint(0, 15, (T, 3), device="cuda", generator=gen, dtype=torch.int32)
    rank3[::5] = 14                                                    # the last row of every positional table
    pl = Layout()
    for name, rows, ld in (("Wg", 128, 8), ("We", 128, ng), ("be", 1, 128), ("E0", 15, 42), ("E1", 15, 42), ("E2", 15, 44)):
        pl.add(name, rows, ld)
    P = pl.build(nb)
    sl = Layout()
    for name, ld in (("V0", 24), ("GD", 6), ("SH", KS), ("VG", 384), ("H", 256)):
        sl.add(name, T, ld)
    S = sl.build(nb)
    shapes = {"Wg": (128, 8), "We": (128, ng), "be": (1, 128), "E0": (15, 42), "E1": (15, 42), "E2": (15, 44)}
    for z in range(nb):
        for name, (rows, cols) in shapes.items():
            P.view(z, rows, cols, cols, pl.off[name]).copy_(rnd(gen, rows, cols, 0.3))
    want = Want(S)
    for z in range(nb):
        b = z % in_nets
        pr = {k: P.view(z, *shapes[k], shapes[k][1], pl.off[k]) for k in shapes}
        ref = R.embed_fwd_ref(obs.view(b, T, 41, 41), act.view(b, T, 3, 3) if act else None, rank3, pr["Wg"], pr["We"], pr["be"][0],
                              pr["E0"], pr["E1"], pr["E2"])
        for name, cols, ld, off in (("V0", 24, 24, sl.off["V0"]), ("GD", 6, 6, sl.off["GD"]), ("SH", ng, KS, sl.off["SH"]),
                                    ("VG", 384, 384, sl.off["VG"]), ("H", 128, 256, sl.off["H"] + 128)):
            want.set(z, T, cols, ld, off, ref[name][0], ref[name][1])
    g = call("sgrl_embed_fwd", obs.ptr(), obs.zs, act.ptr() if act else None, act.zs if act else 0, rank3.data_ptr(),
             *(P.ptr(pl.off[k]) for k in shapes), P.zs, S.ptr(sl.off["V0"]), S.ptr(sl.off["GD"]), S.ptr(sl.off["SH"]), KS,
             S.ptr(sl.off["VG"]), S.ptr(sl.off["H"] + 128), 256, S.zs, T, ng, nb, in_nets)
    gx = min(max((T + 7) // 8, 1), EMBED_CAP)
    r.grid("embed_fwd", ("walk" if (T + 7) // 8 > EMBED_CAP else "group-per-cta") + ("+partial-group" if T % 8 else ""), g, (gx, nb, 1))
    r.regimes.add(("embed_fwd", f"in_nets={'nb' if in_nets == nb else '<nb'}"))
    # V0, GD and SH are copies: bit for bit (scale 0); VG and H within their scales
    _split_check(r, want, "embed_fwd", {name: [(off, T, cols, ld)] for name, cols, ld, off in (
        ("V0", 24, 24, sl.off["V0"]), ("GD", 6, 6, sl.off["GD"]), ("SH", ng, KS, sl.off["SH"]), ("VG", 384, 384, sl.off["VG"]),
        ("H", 128, 256, sl.off["H"] + 128))})


# ================================================================================================================= input_grad
def ragged_sizes(gen, T):
    """graph sizes 2..16 in random order summing to T, with at least one 16-limb and one 2-limb graph (T = 1: one token)."""
    sizes = [16, 2] if T >= 18 else []
    left = T - sum(sizes)
    while left > 0:
        n = min(int(torch.randint(2, 17, (1,), generator=gen)), left)
        if left - n == 1:                                  # never leave a single token behind
            n = n - 1 if n > 2 else n + 1
        sizes.append(n)
        left -= n
    assert sum(sizes) == T and all(n <= 16 for n in sizes) and (T == 1 or min(sizes) >= 2), sizes
    perm = torch.randperm(len(sizes), generator=gen).tolist()
    return [sizes[i] for i in perm]


def input_grad_case(r, T, L, kind, nb, seed, deterministic=False):
    cpu = torch.Generator().manual_seed(seed)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    actor = kind == "actor"
    ng, KS, ma = (17, 145, 0.4) if actor else (20, 148, 1.0)
    sizes = ragged_sizes(cpu, T)
    cu = torch.tensor([0] + torch.tensor(sizes).cumsum(0).tolist(), dtype=torch.int32, device="cuda")
    wl, sl, pl = Layout(), Layout(), Layout()
    for name, ld in (("dvg0", 384), ("dh0", 128), ("dzh", 96), ("dzh2", 96), ("dsh", KS)):
        wl.add(name, T, ld)
    for s in range(3 * L):
        wl.add(f"dz{s}", T, 96)
    for l in range(L):
        wl.add(f"dog{l}", T, 768)
        sl.add(f"P{l}", T, 32)
    sl.add("out", T, 3)
    sl.add("w3", T, 3)
    for name, rows, ld in (("Wg", 128, 8), ("We", 128, ng), ("gg", 30, 136), ("gph", 30, 136)):
        pl.add(name, rows, ld)
    W, S, P = wl.build(nb), sl.build(nb), pl.build(nb)
    dout, dobs = Buf(nb, 3 * T), Buf(nb, 41 * T)
    # P[i][h][j] for j past the query's graph is never read: NaN there
    jmask = torch.zeros(T, 2, 16, dtype=torch.bool, device="cuda")
    for g0, n in zip(cu[:-1].tolist(), sizes):
        jmask[g0:g0 + n, :, :n] = True
    for z in range(nb):
        for name, ld in (("dvg0", 384), ("dh0", 128), ("dzh", 96), ("dzh2", 96), ("dsh", KS)):
            W.view(z, T, ld, ld, wl.off[name]).copy_(rnd(gen, T, ld))
        for s in range(3 * L):
            W.view(z, T, 96, 96, wl.off[f"dz{s}"]).copy_(rnd(gen, T, 96))
        for l in range(L):
            W.view(z, T, 768, 768, wl.off[f"dog{l}"]).copy_(rnd(gen, T, 768))
            pv = torch.rand(T, 2, 16, device="cuda", generator=gen)
            S.view(z, T, 32, 32, sl.off[f"P{l}"]).copy_(torch.where(jmask, pv, torch.full_like(pv, NAN)).view(T, 32))
        p = rnd(gen, T, 3, 3.0)
        p[::7] *= 10.0                                                         # saturated tanh
        S.view(z, T, 3, 3, sl.off["out"]).copy_(ma * torch.tanh(p))
        S.view(z, T, 3, 3, sl.off["w3"]).copy_(rnd(gen, T, 3))
        for name, rows, cols in (("Wg", 128, 8), ("We", 128, ng), ("gg", 30, 136), ("gph", 30, 136)):
            P.view(z, rows, cols, cols, pl.off[name]).copy_(rnd(gen, rows, cols, 0.3))
        dout.view(z, T, 3, 3).copy_(rnd(gen, T, 3))
    want = Want(dobs)
    for z in range(nb):
        v = lambda b, name, ld, off: b.view(z, T, ld, ld, off[name])
        ref = R.input_grad_ref(v(W, "dvg0", 384, wl.off), v(W, "dh0", 128, wl.off), v(W, "dzh", 96, wl.off),
                               v(W, "dzh2", 96, wl.off) if actor else None, v(W, "dsh", KS, wl.off),
                               [v(W, f"dz{s}", 96, wl.off) for s in range(3 * L)], [v(W, f"dog{l}", 768, wl.off) for l in range(L)],
                               [torch.nan_to_num(v(S, f"P{l}", 32, sl.off)) for l in range(L)],
                               P.view(z, 128, 8, 8, pl.off["Wg"]), P.view(z, 128, ng, ng, pl.off["We"]), P.view(z, 30, 136, 136, pl.off["gg"]),
                               P.view(z, 30, 136, 136, pl.off["gph"]) if actor else None, dout.view(z, T, 3, 3) if actor else None,
                               v(S, "out", 3, sl.off) if actor else None, v(S, "w3", 3, sl.off), ma, cu, L)
        want.set(z, T, 41, 41, 0, *ref["dobs"])
    arr = lambda xs: (C.c_void_p * len(xs))(*xs)
    dz = arr([W.ptr(wl.off[f"dz{s}"]) for s in range(3 * L)])
    dog = arr([W.ptr(wl.off[f"dog{l}"]) for l in range(L)])
    Pp = arr([S.ptr(sl.off[f"P{l}"]) for l in range(L)])
    prev = det(deterministic)
    try:
        outs = []
        for _ in range(2):
            dobs.t.copy_(want.before)
            g = call("sgrl_input_grad", W.ptr(wl.off["dvg0"]), W.ptr(wl.off["dh0"]), W.ptr(wl.off["dzh"]),
                     W.ptr(wl.off["dzh2"]) if actor else None, W.ptr(wl.off["dsh"]), KS, dz, dog, Pp, P.ptr(pl.off["Wg"]),
                     P.ptr(pl.off["We"]), P.ptr(pl.off["gg"]), P.ptr(pl.off["gph"]) if actor else None, ng,
                     dout.ptr() if actor else None, dout.zs, S.ptr(sl.off["out"]) if actor else None,
                     S.ptr(sl.off["w3"]) if actor else None, ma, dobs.ptr(), dobs.zs, cu.data_ptr(), len(sizes), T, L, W.zs, S.zs, P.zs, nb)
            outs.append(dobs.t.clone())
    finally:
        det(prev)
    assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32)), "input_grad: two runs differ"
    r.grid("input_grad", warp_regime(T, BWD_CAP), g, (warp_grid(T, BWD_CAP), nb, 1))
    r.regimes.add(("input_grad", f"{kind}-L{L}"))
    r.check("input_grad.dobs", want)


# ================================================================================================================= pos_embed_bwd
def pos_embed_case(r, T, nb, ldh, seed, deterministic=False):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    W = Buf(nb, T * ldh)
    gl = Layout()
    for i, w in enumerate((42, 42, 44)):
        gl.add(f"E{i}", 15, w)
    Gd = gl.build(nb)
    rank3 = torch.randint(0, 15, (T, 3), device="cuda", generator=gen, dtype=torch.int32)
    rank3[::3, 1] = 14
    for z in range(nb):
        W.view(z, T, 128, ldh).copy_(rnd(gen, T, 128))
        for i, w in enumerate((42, 42, 44)):
            Gd.view(z, 15, w, w, gl.off[f"E{i}"]).copy_(rnd(gen, 15, w))
    want = Want(Gd)
    for z in range(nb):
        ref = R.pos_embed_bwd_ref(W.view(z, T, 128, ldh), rank3)
        for i, w in enumerate((42, 42, 44)):
            want.set(z, 15, w, w, gl.off[f"E{i}"], *ref[f"dE{i}"], acc=True)
    prev = det(deterministic)
    try:
        outs = []
        for _ in range(2 if deterministic else 1):
            Gd.t.copy_(want.before)
            g = call("sgrl_pos_embed_bwd", W.ptr(), ldh, W.zs, rank3.data_ptr(), *(Gd.ptr(gl.off[f"E{i}"]) for i in range(3)), Gd.zs, T, nb)
            outs.append(Gd.t.clone())
    finally:
        det(prev)
    gx = 1 if deterministic else min(max((T + 63) // 64, 1), 148)
    reg = "single-cta" if deterministic else ("148-ranges" if (T + 63) // 64 >= 148 else "64-token-ranges")
    r.grid("pos_embed_bwd", reg, g, (gx, nb, 1))
    if deterministic:
        assert (T + 63) // 64 > 1 and torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    r.check("pos_embed_bwd.dE", want)


# ================================================================================================================= layernorm
def ln_rows(gen, T, scale=1.0):
    """LayerNorm inputs: random rows, every 5th with mean 1e3 and std 1e-2, every 7th constant (var = 0)."""
    a = rnd(gen, T, 128, scale)
    a[1::5] = rnd(gen, len(range(1, T, 5)), 128, 1e-2, 1e3)
    a[3::7] = rnd(gen, len(range(3, T, 7)), 1)
    return a


def layernorm_fwd_case(r, T, nb, resid, vec, y2, seed):
    """vec: a, b, y (and y2) on the float4 path (the layers' LN1 / LN2 layout); else scalar (odd offsets or row strides: the
    actor's final norm writes y into SH + 17 with row stride 145, next to s0 in columns 0..16)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    lda, aoff = (256, 128) if vec else (129, 1)
    ldb, boff = (128, 0) if vec else (131, 3)
    ldy, yoff = (256, 128) if vec else (145, 17)
    sl = Layout()
    sl.add("a", T, lda)
    sl.add("b", T, ldb)
    sl.add("x", T, 128)
    sl.add("y", T, ldy)
    sl.add("y2", T, ldy)
    sl.add("st", T, 2)
    S = sl.build(nb)
    pl = Layout()
    pl.add("g", 1, 128)
    pl.add("be", 1, 128)
    P = pl.build(nb)
    for z in range(nb):
        S.view(z, T, 128, lda, sl.off["a"] + aoff).copy_(ln_rows(gen, T))
        if resid:
            S.view(z, T, 128, ldb, sl.off["b"] + boff).copy_(rnd(gen, T, 128, 1e-3))
        S.view(z, T, yoff, ldy, sl.off["y"]).copy_(rnd(gen, T, yoff))        # s0 (and the left half of u): must survive the store
        P.view(z, 1, 128, 128, pl.off["g"]).copy_(rnd(gen, 1, 128, 0.5, 1.0))
        P.view(z, 1, 128, 128, pl.off["be"]).copy_(rnd(gen, 1, 128, 0.5))
    want = Want(S)
    for z in range(nb):
        ref = R.layernorm_fwd_ref(S.view(z, T, 128, lda, sl.off["a"] + aoff), S.view(z, T, 128, ldb, sl.off["b"] + boff) if resid else None,
                                  P.view(z, 1, 128, 128, pl.off["g"])[0], P.view(z, 1, 128, 128, pl.off["be"])[0])
        want.set(z, T, 128, 128, sl.off["x"], *ref["x"])
        want.set(z, T, 128, ldy, sl.off["y"] + yoff, *ref["y"])
        if y2:
            want.set(z, T, 128, ldy, sl.off["y2"] + yoff, *ref["y"])
        want.set(z, T, 1, 2, sl.off["st"], *ref["mean"])
        want.set(z, T, 1, 2, sl.off["st"] + 1, *ref["rstd"])
    g = call("sgrl_layernorm_fwd", S.ptr(sl.off["a"] + aoff), lda, S.ptr(sl.off["b"] + boff) if resid else None, ldb,
             P.ptr(pl.off["g"]), P.ptr(pl.off["be"]), P.zs, S.ptr(sl.off["x"]), S.ptr(sl.off["y"] + yoff), ldy,
             S.ptr(sl.off["y2"] + yoff) if y2 else None, ldy, S.ptr(sl.off["st"]), S.zs, T, nb)
    r.grid("layernorm_fwd", warp_regime(T), g, (warp_grid(T), nb, 1))
    r.regimes.add(("layernorm_fwd", "float4" if vec else "scalar"))
    # one measure per output class: x, y (+ y2), stats
    _split_check(r, want, "layernorm_fwd", {"x": [(sl.off["x"], T, 128, 128)],
                                            "y": [(sl.off["y"] + yoff, T, 128, ldy)] + ([(sl.off["y2"] + yoff, T, 128, ldy)] if y2 else []),
                                            "stats": [(sl.off["st"], T, 2, 2)]})


def _split_check(r, want, kernel, parts):
    """the sentinels of the whole buffer, then the worst ratio of each named group of regions"""
    want.measure(kernel)
    for name, regions in parts.items():
        mask = torch.zeros_like(want.mask)
        for off, rows, cols, ld in regions:
            for z in range(want.buf.nb):
                mask.as_strided((rows, cols), (ld, 1), z * want.buf.zs + off).fill_(True)
        w, where = want.worst(mask & want.mask)
        if w is not None:
            r.ratios.append((f"{kernel}.{name}", w, where))


def layernorm_bwd_case(r, T, nb, vec, dy2, wgrad, tail, seed, deterministic=False):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    # float4: the layers' LN2 / LN1 layout; scalar: the actor's final norm reads dy from W_DSH + 17 (row stride 145), plus odd
    # offsets for every other operand
    ld1, o1 = (128, 0) if vec else (145, 17)
    ld2, o2 = (256, 128) if vec else (257, 129)
    ldx, ox = (128, 0) if vec else (129, 1)
    lddx, odx = (128, 0) if vec else (131, 2)
    ldry, ory = (128, 0) if vec else (133, 3)
    ldro, oro = (128, 0) if vec else (130, 1)
    wl, sl, gl, pl = Layout(), Layout(), Layout(), Layout()
    for name, ld in (("dy1", ld1), ("dy2", ld2), ("dx", lddx), ("ro", ldro)):
        wl.add(name, T, ld)
    wl.add("dF", T, 1)
    for name, ld in (("x", ldx), ("ry", ldry)):
        sl.add(name, T, ld)
    sl.add("st", T, 2)
    sl.add("F", T, 1)
    pl.add("g", 1, 128)
    gl.add("dg", 1, 128)
    gl.add("db", 1, 128)
    W, S, P, Gd = wl.build(nb), sl.build(nb), pl.build(nb), gl.build(nb)
    for z in range(nb):
        W.view(z, T, 128, ld1, wl.off["dy1"] + o1).copy_(rnd(gen, T, 128))
        if dy2:
            W.view(z, T, 128, ld2, wl.off["dy2"] + o2).copy_(rnd(gen, T, 128))
        x = ln_rows(gen, T)
        S.view(z, T, 128, ldx, sl.off["x"] + ox).copy_(x)
        f = R.layernorm_fwd_ref(x, None, torch.ones(128, device="cuda"), torch.zeros(128, device="cuda"))
        S.view(z, T, 2, 2, sl.off["st"]).copy_(torch.stack([f["mean"][0], f["rstd"][0]], 1))
        P.view(z, 1, 128, 128, pl.off["g"]).copy_(rnd(gen, 1, 128, 0.5, 1.0))
        Gd.view(z, 1, 128, 128, gl.off["dg"]).copy_(rnd(gen, 1, 128))
        Gd.view(z, 1, 128, 128, gl.off["db"]).copy_(rnd(gen, 1, 128))
        if tail:
            S.view(z, T, 128, ldry, sl.off["ry"] + ory).copy_(rnd(gen, T, 128))
            S.view(z, T, 1, 1, sl.off["F"]).copy_(f_divisors(gen, T)[:, None])
            W.view(z, T, 1, 1, wl.off["dF"]).copy_(rnd(gen, T, 1))
    wW, wG = Want(W), Want(Gd)
    for z in range(nb):
        ref = R.layernorm_bwd_ref(W.view(z, T, 128, ld1, wl.off["dy1"] + o1), W.view(z, T, 128, ld2, wl.off["dy2"] + o2) if dy2 else None,
                                  S.view(z, T, 128, ldx, sl.off["x"] + ox), S.view(z, T, 2, 2, sl.off["st"]), P.view(z, 1, 128, 128, pl.off["g"])[0],
                                  S.view(z, T, 128, ldry, sl.off["ry"] + ory) if tail else None, S.view(z, T, 1, 1, sl.off["F"]) if tail else None)
        wW.set(z, T, 128, lddx, wl.off["dx"] + odx, *ref["dx"])
        if tail:
            wW.set(z, T, 128, ldro, wl.off["ro"] + oro, *ref["rd_out"])
            wW.set(z, T, 1, 1, wl.off["dF"], *ref["rd_dF"], acc=True)
        if wgrad:
            wG.set(z, 1, 128, 128, gl.off["dg"], *ref["dgamma"], acc=True)
            wG.set(z, 1, 128, 128, gl.off["db"], *ref["dbeta"], acc=True)
    prev = det(deterministic)
    try:
        outs = []
        for _ in range(2 if deterministic else 1):
            W.t.copy_(wW.before)
            Gd.t.copy_(wG.before)
            g = call("sgrl_layernorm_bwd", W.ptr(wl.off["dy1"] + o1), ld1, W.ptr(wl.off["dy2"] + o2) if dy2 else None, ld2,
                     S.ptr(sl.off["x"] + ox), ldx, S.ptr(sl.off["st"]), S.zs, P.ptr(pl.off["g"]), P.zs, W.ptr(wl.off["dx"] + odx), lddx, W.zs,
                     Gd.ptr(gl.off["dg"]) if wgrad else None, Gd.ptr(gl.off["db"]) if wgrad else None, Gd.zs,
                     S.ptr(sl.off["ry"] + ory) if tail else None, ldry, S.ptr(sl.off["F"]) if tail else None,
                     W.ptr(wl.off["dF"]) if tail else None, W.ptr(wl.off["ro"] + oro) if tail else None, ldro, T, nb)
            outs.append((W.t.clone(), Gd.t.clone()))
    finally:
        det(prev)
    single = deterministic and wgrad
    r.grid("layernorm_bwd", "single-cta" if single else warp_regime(T, BWD_CAP), g, (1 if single else warp_grid(T, BWD_CAP), nb, 1))
    r.regimes.add(("layernorm_bwd", ("float4" if vec else "scalar") + ("+tail" if tail else "") + ("+wgrad" if wgrad else "")))
    if deterministic:
        assert warp_grid(T, BWD_CAP) > 1
        for a, b in zip(*outs):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "layernorm_bwd: deterministic runs differ"
    _split_check(r, wW, "layernorm_bwd", {"dx": [(wl.off["dx"] + odx, T, 128, lddx)], "rd_out": [(wl.off["ro"] + oro, T, 128, ldro)],
                                          "rd_dF": [(wl.off["dF"], T, 1, 1)]})
    _split_check(r, wG, "layernorm_bwd", {"dgamma": [(gl.off["dg"], 1, 128, 128), (gl.off["db"], 1, 128, 128)]})


# ================================================================================================================= matrix apply
def matapply_case(r, T, nb, which, seed, keep_r=True):
    """which: fwd | bwd | l5_fwd | l5_bwd"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    sl, wl, pl = Layout(), Layout(), Layout()
    for name, ld in (("Z", 96), ("M", 1024), ("F", 1), ("R", 96), ("Vg", 384), ("dV", 384), ("Vn", 384)):
        sl.add(name, T, ld)
    for name, ld in (("dR", 96), ("dVn", 384), ("dZ", 96), ("dT", 1024), ("dF", 1)):
        wl.add(name, T, ld)
    pl.add("W5", 128, 32)
    S, Wk, P = sl.build(nb), wl.build(nb), pl.build(nb)
    for z in range(nb):
        S.view(z, T, 96, 96, sl.off["Z"]).copy_(rnd(gen, T, 96))
        F = f_divisors(gen, T)
        S.view(z, T, 1024, 1024, sl.off["M"]).copy_(rnd(gen, T, 1024) / F[:, None])
        S.view(z, T, 1, 1, sl.off["F"]).copy_(F[:, None])
        P.view(z, 128, 32, 32, pl.off["W5"]).copy_(rnd(gen, 128, 32, 0.2))
        for name, ld in (("Vg", 384), ("dV", 384)):
            S.view(z, T, ld, ld, sl.off[name]).copy_(rnd(gen, T, ld))
        for name, ld in (("dR", 96), ("dVn", 384), ("dF", 1)):
            Wk.view(z, T, ld, ld, wl.off[name]).copy_(rnd(gen, T, ld))
    wS, wW = Want(S), Want(Wk)
    v = lambda b, off, z, name, ld: b.view(z, T, ld, ld, off[name])
    for z in range(nb):
        Z, M, F = v(S, sl.off, z, "Z", 96), v(S, sl.off, z, "M", 1024), v(S, sl.off, z, "F", 1)
        if which == "fwd":
            wS.set(z, T, 96, 96, sl.off["R"], *R.matapply_fwd_ref(Z, M)["R"])
        elif which == "l5_fwd":
            ref = R.matapply_l5_fwd_ref(Z, M, P.view(z, 128, 32, 32, pl.off["W5"]), v(S, sl.off, z, "Vg", 384), v(S, sl.off, z, "dV", 384))
            if keep_r:
                wS.set(z, T, 96, 96, sl.off["R"], *ref["R"])
            wS.set(z, T, 384, 384, sl.off["Vn"], *ref["Vn"])
        else:
            ref = R.matapply_bwd_ref(v(Wk, wl.off, z, "dR", 96), Z, M, F) if which == "bwd" else \
                R.matapply_l5_bwd_ref(v(Wk, wl.off, z, "dVn", 384), P.view(z, 128, 32, 32, pl.off["W5"]), Z, M, F)
            wW.set(z, T, 96, 96, wl.off["dZ"], *ref["dZ"])
            wW.set(z, T, 1024, 1024, wl.off["dT"], *ref["dT"])
            wW.set(z, T, 1, 1, wl.off["dF"], *ref["dF"], acc=True)
    s, w = S.ptr, Wk.ptr
    if which == "fwd":
        g = call("sgrl_matapply_fwd", s(sl.off["Z"]), s(sl.off["M"]), s(sl.off["R"]), S.zs, T, nb)
    elif which == "bwd":
        g = call("sgrl_matapply_bwd", w(wl.off["dR"]), s(sl.off["Z"]), s(sl.off["M"]), s(sl.off["F"]), S.zs, w(wl.off["dZ"]), w(wl.off["dT"]),
                 w(wl.off["dF"]), Wk.zs, T, nb)
    elif which == "l5_fwd":
        g = call("sgrl_matapply_l5_fwd", s(sl.off["Z"]), s(sl.off["M"]), P.ptr(pl.off["W5"]), P.zs, s(sl.off["Vg"]), s(sl.off["dV"]),
                 s(sl.off["R"]) if keep_r else None, s(sl.off["Vn"]), S.zs, T, nb)
    else:
        g = call("sgrl_matapply_l5_bwd", w(wl.off["dVn"]), P.ptr(pl.off["W5"]), P.zs, s(sl.off["Z"]), s(sl.off["M"]), s(sl.off["F"]), S.zs,
                 w(wl.off["dZ"]), w(wl.off["dT"]), w(wl.off["dF"]), Wk.zs, T, nb)
    kern = f"matapply_{which}"
    r.grid(kern, warp_regime(T), g, (warp_grid(T), nb, 1))
    if which == "l5_fwd":
        r.regimes.add((kern, "R kept" if keep_r else "R null"))
    if which in ("fwd", "l5_fwd"):
        _split_check(r, wS, kern, {"R": [(sl.off["R"], T, 96, 96)], **({"Vn": [(sl.off["Vn"], T, 384, 384)]} if which == "l5_fwd" else {})})
        wW.measure(kern)
    else:
        _split_check(r, wW, kern, {"dZ": [(wl.off["dZ"], T, 96, 96)], "dT": [(wl.off["dT"], T, 1024, 1024)], "dF": [(wl.off["dF"], T, 1, 1)]})
        wS.measure(kern)


# ================================================================================================================= actor head
def actor_out_case(r, T, nb, bwd, max_action, seed, deterministic=False):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    sl, wl, pl, gl = Layout(), Layout(), Layout(), Layout()
    for name, ld in (("R", 96), ("V0", 24), ("W3", 3), ("out", 3)):
        sl.add(name, T, ld)
    wl.add("dR", T, 96)
    pl.add("wd", 1, 32)
    gl.add("dwd", 1, 32)
    S, Wk, P, Gd = sl.build(nb), wl.build(nb), pl.build(nb), gl.build(nb)
    dout = Buf(nb, 3 * T)
    for z in range(nb):
        S.view(z, T, 96, 96, sl.off["R"]).copy_(rnd(gen, T, 96))
        V0 = rnd(gen, T, 24)
        V0[::4] *= 30.0                                                    # |p| > 10: saturated tanh
        S.view(z, T, 24, 24, sl.off["V0"]).copy_(V0)
        P.view(z, 1, 32, 32, pl.off["wd"]).copy_(rnd(gen, 1, 32, 0.3))
        Gd.view(z, 1, 32, 32, gl.off["dwd"]).copy_(rnd(gen, 1, 32))
        dout.view(z, T, 3, 3).copy_(rnd(gen, T, 3))
        if bwd:      # the forward's out, as the kernel stored it
            f = R.actor_out_fwd_ref(S.view(z, T, 96, 96, sl.off["R"]), S.view(z, T, 24, 24, sl.off["V0"]), P.view(z, 1, 32, 32, pl.off["wd"]), max_action)
            S.view(z, T, 3, 3, sl.off["out"]).copy_(f["out"][0].float())
    wS, wW, wG = Want(S), Want(Wk), Want(Gd)
    for z in range(nb):
        Rz, V0z, wd = S.view(z, T, 96, 96, sl.off["R"]), S.view(z, T, 24, 24, sl.off["V0"]), P.view(z, 1, 32, 32, pl.off["wd"])
        if bwd:
            ref = R.actor_out_bwd_ref(dout.view(z, T, 3, 3), S.view(z, T, 3, 3, sl.off["out"]), Rz, V0z, wd, max_action)
            wW.set(z, T, 96, 96, wl.off["dR"], *ref["dR"])
            wG.set(z, 1, 32, 32, gl.off["dwd"], *ref["dwd"], acc=True)
        else:
            ref = R.actor_out_fwd_ref(Rz, V0z, wd, max_action)
            wS.set(z, T, 3, 3, sl.off["W3"], *ref["W3"])
            wS.set(z, T, 3, 3, sl.off["out"], *ref["out"])
    prev = det(deterministic)
    try:
        outs = []
        for _ in range(2 if deterministic else 1):
            Wk.t.copy_(wW.before)
            Gd.t.copy_(wG.before)
            if bwd:
                g = call("sgrl_actor_out_bwd", dout.ptr(), dout.zs, S.ptr(sl.off["out"]), S.ptr(sl.off["R"]), S.ptr(sl.off["V0"]), S.zs,
                         P.ptr(pl.off["wd"]), P.zs, Wk.ptr(wl.off["dR"]), Wk.zs, Gd.ptr(gl.off["dwd"]), Gd.zs, max_action, T, nb)
            else:
                g = call("sgrl_actor_out_fwd", S.ptr(sl.off["R"]), S.ptr(sl.off["V0"]), P.ptr(pl.off["wd"]), P.zs, S.ptr(sl.off["W3"]),
                         S.ptr(sl.off["out"]), S.zs, max_action, T, nb)
            outs.append((Wk.t.clone(), Gd.t.clone()))
    finally:
        det(prev)
    if bwd:
        r.grid("actor_out_bwd", "single-cta" if deterministic else warp_regime(T, BWD_CAP), g,
               (1 if deterministic else warp_grid(T, BWD_CAP), nb, 1))
        if deterministic:
            assert warp_grid(T, BWD_CAP) > 1
            for a, b in zip(*outs):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "actor_out_bwd: deterministic runs differ"
        _split_check(r, wW, "actor_out_bwd", {"dR": [(wl.off["dR"], T, 96, 96)]})
        _split_check(r, wG, "actor_out_bwd", {"dwd": [(gl.off["dwd"], 1, 32, 32)]})
        wS.measure("actor_out_bwd")
    else:
        r.grid("actor_out_fwd", warp_regime(T), g, (warp_grid(T), nb, 1))
        _split_check(r, wS, "actor_out_fwd", {"W3": [(sl.off["W3"], T, 3, 3)], "out": [(sl.off["out"], T, 3, 3)]})


# ================================================================================================================= rowdiv_bwd
def rowdiv_case(r, T, nb, variant, seed):
    """qkv: N = 768, q columns scaled, in place; critic: N = 1 from dOut (src) into a dy of row stride 4; dff: N = 128 from dx (src)"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    N, cs, cs_n, lddy, ldsrc, src = {"qkv": (768, 0.08838834764831845, 256, 768, 0, False), "critic": (1, 1.0, 0, 4, 1, True),
                                     "dff": (128, 1.0, 0, 128, 128, True)}[variant]
    wl, sl = Layout(), Layout()
    wl.add("dy", T, lddy)
    wl.add("dF", T, 1)
    sl.add("y", T, N)
    sl.add("F", T, 1)
    Wk, S = wl.build(nb), sl.build(nb)
    Sr = Buf(nb, T * max(ldsrc, 1)) if src else None
    for z in range(nb):
        g_in = rnd(gen, T, N)
        (Sr.view(z, T, N, ldsrc) if src else Wk.view(z, T, N, lddy, wl.off["dy"])).copy_(g_in)
        S.view(z, T, N, N, sl.off["y"]).copy_(rnd(gen, T, N))
        S.view(z, T, 1, 1, sl.off["F"]).copy_(f_divisors(gen, T)[:, None])
        Wk.view(z, T, 1, 1, wl.off["dF"]).copy_(rnd(gen, T, 1))
    wW = Want(Wk)
    for z in range(nb):
        g_in = Sr.view(z, T, N, ldsrc) if src else Wk.view(z, T, N, lddy, wl.off["dy"])
        ref = R.rowdiv_bwd_ref(g_in, S.view(z, T, N, N, sl.off["y"]), S.view(z, T, 1, 1, sl.off["F"]), cs, cs_n)
        wW.set(z, T, N, lddy, wl.off["dy"], *ref["dt"])
        wW.set(z, T, 1, 1, wl.off["dF"], *ref["dF"], acc=True)
    g = call("sgrl_rowdiv_bwd", Wk.ptr(wl.off["dy"]), lddy, Wk.zs, S.ptr(sl.off["y"]), N, S.ptr(sl.off["F"]), S.zs, Wk.ptr(wl.off["dF"]), N,
             cs, cs_n, Sr.ptr() if src else None, ldsrc, Sr.zs if src else 0, T, nb)
    r.grid("rowdiv_bwd", warp_regime(T), g, (warp_grid(T), nb, 1))
    r.regimes.add(("rowdiv_bwd", variant))
    _split_check(r, wW, "rowdiv_bwd", {"dt": [(wl.off["dy"], T, N, lddy)], "dF": [(wl.off["dF"], T, 1, 1)]})


# ================================================================================================================= colsum
def colsum_case(r, M, N, nb, seed, deterministic=False):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    ldx = N + 5
    X, O = Buf(nb, M * ldx), Buf(nb, N + 7)
    for z in range(nb):
        X.view(z, M, N, ldx).copy_(rnd(gen, M, N))
        O.view(z, 1, N, N).copy_(rnd(gen, 1, N))
    want = Want(O)
    for z in range(nb):
        want.set(z, 1, N, N, 0, *R.colsum_ref(X.view(z, M, N, ldx), -0.75)["out"], acc=True)
    prev = det(deterministic)
    try:
        outs = []
        for _ in range(2 if deterministic else 1):
            O.t.copy_(want.before)
            g = call("sgrl_colsum", X.ptr(), ldx, X.zs, O.ptr(), O.zs, M, N, -0.75, nb)
            outs.append(O.t.clone())
    finally:
        det(prev)
    gy = 1 if deterministic else min(max((M + 63) // 64, 1), 32)
    r.grid("colsum", "single-slice" if deterministic else ("y-split-32" if gy == 32 else "y-split<32"), g, ((N + 31) // 32, gy, nb))
    r.regimes.add(("colsum", f"N={N}"))
    if deterministic:
        assert min(max((M + 63) // 64, 1), 32) > 1
        assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32)), "colsum: deterministic runs differ"
    r.check("colsum.out", want)


# ================================================================================================================= block_copy
def block_copy_case(r, M, N, nb, add, two, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    ldd, lds, lds2 = N + 3, N + 1, N + 6
    D, S1, S2 = Buf(nb, M * ldd), Buf(nb, M * lds), Buf(nb, M * lds2)
    for z in range(nb):
        D.view(z, M, N, ldd).copy_(rnd(gen, M, N))
        S1.view(z, M, N, lds).copy_(rnd(gen, M, N))
        S2.view(z, M, N, lds2).copy_(rnd(gen, M, N))
    want = Want(D)
    for z in range(nb):
        v = S1.view(z, M, N, lds)
        if two:
            v = v + S2.view(z, M, N, lds2)
        if add:
            v = D.view(z, M, N, ldd) + v
        want.set(z, M, N, ldd, 0, v)
    g = call("sgrl_block_copy", D.ptr(), ldd, D.zs, S1.ptr(), lds, S1.zs, S2.ptr() if two else None, lds2, S2.zs, M, N, add, nb)
    gx = min(max((M * N + 255) // 256, 1), EMBED_CAP)
    r.grid("block_copy", "walk" if (M * N + 255) // 256 > EMBED_CAP else "element-per-thread", g, (gx, nb, 1))
    r.check("block_copy", want)


# ================================================================================================================= fold / unfold
def fold_case(r, L, nb, with_split, seed, unfold=False):
    """The network's n = 2L + 1 folds: (256,1024) weights of every layer, then the head's (128,1024)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rows = [256] * (2 * L) + [128]
    n = len(rows)
    src = [sum(rw * 1024 + 64 for rw in rows[:i]) + 16 for i in range(n)]          # not packed back to back: gaps stay sentinels
    dst = [sum(rw * GP_K for rw in rows[:i]) for i in range(n)]
    plane = r4(sum(rw * GP_K for rw in rows)) + 32
    big = Buf(nb, src[-1] + rows[-1] * 1024 + 64)                                   # params (fold) / gradients (unfold)
    fb = Buf(nb, 3 * plane)                                                         # fold planes (fold) / folded gradients (unfold)
    slots = pack_indices()[0]
    pad = torch.tensor(sorted(set(range(GP_K)) - set(slots)), device="cuda")
    for z in range(nb):
        for m in range(n):
            big.view(z, rows[m], 1024, 1024, src[m]).copy_(rnd(gen, rows[m], 1024))
            if unfold:
                gf = rnd(gen, rows[m], GP_K)
                gf[:, pad] = NAN                                                    # never read
                fb.view(z, rows[m], GP_K, GP_K, dst[m]).copy_(gf)
    out = big if unfold else fb
    want = Want(out)
    for z in range(nb):
        for m in range(n):
            if unfold:
                t = R.unfold_ref(fb.view(z, rows[m], GP_K, GP_K, dst[m]))
                want.set(z, rows[m], 1024, 1024, src[m], big.view(z, rows[m], 1024, 1024, src[m]) + t)
            else:
                wf = R.fold_ref(big.view(z, rows[m], 1024, 1024, src[m]))
                want.set(z, rows[m], GP_K, GP_K, dst[m], wf)
                if with_split:
                    hi = _rna_tf32(wf)
                    want.set(z, rows[m], GP_K, GP_K, plane + dst[m], hi)
                    want.set(z, rows[m], GP_K, GP_K, 2 * plane + dst[m], _rna_tf32(wf - hi))
    a64 = lambda xs: (C.c_int64 * n)(*xs)
    if unfold:
        g = call("sgrl_unfold_sym", fb.ptr(), fb.zs, big.ptr(), big.zs, a64(src), a64(dst), (C.c_int32 * n)(*rows), n, nb)
        r.grid("unfold_sym", "64-ctas-per-matrix", g, (64, n, nb))
        r.check("unfold_sym", want)
    else:
        g = call("sgrl_fold_sym", big.ptr(), big.zs, fb.ptr(), fb.zs, plane, with_split, a64(src), a64(dst), (C.c_int32 * n)(*rows), n, nb)
        r.grid("fold_sym", "48-ctas-per-matrix" + ("+tf32-split" if with_split else ""), g, (48, n, nb))
        r.check("fold_sym", want)


def _rna_tf32(x):
    """round-to-nearest, ties away, to 10 mantissa bits (cvt.rna.tf32.f32) with integer ops"""
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


# ================================================================================================================= the cases
CASES = {}


def case(cid, fn, **kw):
    CASES[cid] = (fn, kw)


B256 = 2304                  # tokens per net of the B = 256 humanoid-9 update
ROLL = 147459                # a rollout-size batch (16 384 humanoid-9 graphs + 3 tokens)
for T, nb, inn, kind in ((1, 1, 1, "actor"), (7, 2, 1, "critic"), (2051, 5, 5, "actor"), (B256, 2, 1, "critic"), (4736, 1, 1, "actor"),
                         (4737, 16, 8, "critic"), (4737, 2, 2, "actor"), (ROLL, 1, 1, "actor"), (9472, 16, 16, "critic")):
    case(f"embed-{kind}-T{T}-nb{nb}-in{inn}", embed_case, T=T, nb=nb, in_nets=inn, kind=kind, seed=T + nb)

for T, L, kind, nb in ((1, 1, "actor", 1), (21, 3, "critic", 2), (2051, 8, "actor", 1), (2368, 3, "critic", 5), (2369, 3, "actor", 2),
                       (B256, 3, "actor", 2), (9473, 1, "critic", 1), (9473, 3, "actor", 1)):
    case(f"input_grad-{kind}-T{T}-L{L}-nb{nb}", input_grad_case, T=T, L=L, kind=kind, nb=nb, seed=T + L)
case("input_grad-det-actor-T2369", input_grad_case, T=2369, L=3, kind="actor", nb=2, seed=5, deterministic=True)

for T, nb, ldh in ((1, 1, 128), (7, 2, 256), (2051, 5, 128), (B256, 2, 128), (9472, 1, 128), (9473, 16, 256)):
    case(f"pos_embed_bwd-T{T}-nb{nb}", pos_embed_case, T=T, nb=nb, ldh=ldh, seed=T)
case("pos_embed_bwd-det-T2051", pos_embed_case, T=2051, nb=2, ldh=128, seed=3, deterministic=True)

for T, nb in ((1, 1), (7, 2), (2051, 5), (9472, 1), (9473, 16), (ROLL, 1)):
    for vec in (True, False):
        case(f"layernorm_fwd-{'vec' if vec else 'scalar'}-T{T}-nb{nb}", layernorm_fwd_case, T=T, nb=nb, resid=vec or T % 2 == 1, vec=vec,
             y2=T == 7, seed=T + vec)
case("layernorm_fwd-scalar-final-norm-T2304", layernorm_fwd_case, T=B256, nb=2, resid=False, vec=False, y2=False, seed=1)

for T, nb in ((1, 1), (7, 2), (2051, 5), (2368, 1), (2369, 2), (B256, 16), (9473, 1)):
    for vec in (True, False):
        case(f"layernorm_bwd-{'vec' if vec else 'scalar'}-T{T}-nb{nb}", layernorm_bwd_case, T=T, nb=nb, vec=vec, dy2=vec != (T % 2 == 0),
             wgrad=T != 2368, tail=vec or T == 7, seed=T * 2 + vec)
case("layernorm_bwd-vec-data-only-T2051", layernorm_bwd_case, T=2051, nb=2, vec=True, dy2=True, wgrad=False, tail=False, seed=9)
case("layernorm_bwd-det-vec-T2369", layernorm_bwd_case, T=2369, nb=2, vec=True, dy2=True, wgrad=True, tail=True, seed=4, deterministic=True)
case("layernorm_bwd-det-scalar-T2051", layernorm_bwd_case, T=2051, nb=1, vec=False, dy2=False, wgrad=True, tail=False, seed=6,
     deterministic=True)

for which in ("fwd", "bwd", "l5_fwd", "l5_bwd"):
    for T, nb in ((1, 1), (7, 2), (B256, 5), (9472, 1), (9473, 16)):
        case(f"matapply_{which}-T{T}-nb{nb}", matapply_case, T=T, nb=nb, which=which, seed=T + len(which))
case("matapply_fwd-T147459", matapply_case, T=ROLL, nb=1, which="fwd", seed=2)
case("matapply_l5_fwd-Rnull-T2051", matapply_case, T=2051, nb=2, which="l5_fwd", keep_r=False, seed=3)
case("matapply_l5_fwd-Rnull-T147459", matapply_case, T=ROLL, nb=1, which="l5_fwd", keep_r=False, seed=4)

for T, nb, ma in ((7, 2, 0.4), (B256, 5, 2.5), (9472, 1, 0.4), (9473, 16, 2.5), (ROLL, 1, 1.0)):
    case(f"actor_out_fwd-T{T}-nb{nb}", actor_out_case, T=T, nb=nb, bwd=False, max_action=ma, seed=T)
for T, nb, ma in ((1, 1, 2.5), (2368, 2, 0.4), (2369, 5, 2.5), (9473, 16, 0.4)):
    case(f"actor_out_bwd-T{T}-nb{nb}", actor_out_case, T=T, nb=nb, bwd=True, max_action=ma, seed=T)
case("actor_out_bwd-det-T2051", actor_out_case, T=2051, nb=2, bwd=True, max_action=2.5, seed=8, deterministic=True)

for variant in ("qkv", "critic", "dff"):
    for T, nb in ((1, 1), (7, 2), (B256, 5), (9473, 16)):
        case(f"rowdiv_bwd-{variant}-T{T}-nb{nb}", rowdiv_case, T=T, nb=nb, variant=variant, seed=T + len(variant))

for M, N, nb in ((1, 1, 1), (64, 31, 2), (65, 33, 1), (2047, 1, 5), (2048, 128, 2), (2049, 31, 16), (9473, 33, 1), (B256, 256, 2)):
    case(f"colsum-M{M}-N{N}-nb{nb}", colsum_case, M=M, N=N, nb=nb, seed=M + N)
case("colsum-det-M2049-N33", colsum_case, M=2049, N=33, nb=2, seed=1, deterministic=True)

for M, N, nb, add, two in ((1, 1, 1, 0, False), (7, 3, 2, 0, False), (B256, 3, 5, 1, False), (B256, 128, 2, 0, True),
                           (9473, 128, 16, 1, True)):
    case(f"block_copy-M{M}-N{N}-nb{nb}-add{add}-src2{int(two)}", block_copy_case, M=M, N=N, nb=nb, add=add, two=two, seed=M + N)

for L, nb, split in ((1, 1, 1), (3, 2, 0), (3, 2, 1), (8, 1, 1)):
    case(f"fold_sym-L{L}-nb{nb}-split{split}", fold_case, L=L, nb=nb, with_split=split, seed=L * 4 + split)
for L, nb in ((1, 2), (3, 5), (8, 1)):
    case(f"unfold_sym-L{L}-nb{nb}", fold_case, L=L, nb=nb, with_split=0, seed=L, unfold=True)


class Results(dict):
    """case id -> Run (or the AssertionError it raised, reported by the case's own test), each case run once when first asked
    for: a -k selection runs only its cases, test_regime_coverage all of them."""

    def __missing__(self, cid):
        fn, kw = CASES[cid]
        r = Run()
        try:
            fn(r, **kw)
        except AssertionError as e:
            r = e
        torch.cuda.empty_cache()
        self[cid] = r
        return r


@pytest.fixture(scope="module")
def results():
    return Results()


@pytest.mark.parametrize("cid", list(CASES))
def test_aux_kernel(results, cid):
    r = results[cid]
    if isinstance(r, AssertionError):
        raise r
    for label, w, where in r.ratios:
        print(f"RATIO {cid} {label} {w:.3e} {where}")
        tol = TOL.get(label, 0.0)          # outputs without a tolerance are copies: bit for bit
        assert w <= tol, f"{label}: error {w:.3g} x scale at {where} (tolerance {tol:.2g})"


REGIMES = sorted([
    ("actor_out_bwd", "single-cta"), ("actor_out_bwd", "walk"), ("actor_out_bwd", "warp-per-token"),
    ("actor_out_fwd", "walk"), ("actor_out_fwd", "warp-per-token"),
    ("block_copy", "element-per-thread"), ("block_copy", "walk"),
    ("colsum", "N=1"), ("colsum", "N=31"), ("colsum", "N=33"), ("colsum", "N=128"), ("colsum", "N=256"),
    ("colsum", "single-slice"), ("colsum", "y-split-32"), ("colsum", "y-split<32"),
    ("embed_fwd", "group-per-cta"), ("embed_fwd", "group-per-cta+partial-group"), ("embed_fwd", "walk"), ("embed_fwd", "walk+partial-group"),
    ("embed_fwd", "in_nets=<nb"), ("embed_fwd", "in_nets=nb"),
    ("fold_sym", "48-ctas-per-matrix"), ("fold_sym", "48-ctas-per-matrix+tf32-split"),
    ("input_grad", "actor-L1"), ("input_grad", "actor-L3"), ("input_grad", "actor-L8"), ("input_grad", "critic-L1"), ("input_grad", "critic-L3"),
    ("input_grad", "walk"), ("input_grad", "warp-per-token"),
    ("layernorm_bwd", "float4"), ("layernorm_bwd", "float4+tail"), ("layernorm_bwd", "float4+tail+wgrad"),
    ("layernorm_bwd", "scalar+tail+wgrad"), ("layernorm_bwd", "scalar+wgrad"), ("layernorm_bwd", "scalar"),
    ("layernorm_bwd", "single-cta"), ("layernorm_bwd", "walk"), ("layernorm_bwd", "warp-per-token"),
    ("layernorm_fwd", "float4"), ("layernorm_fwd", "scalar"), ("layernorm_fwd", "walk"), ("layernorm_fwd", "warp-per-token"),
    ("matapply_bwd", "walk"), ("matapply_bwd", "warp-per-token"), ("matapply_fwd", "walk"), ("matapply_fwd", "warp-per-token"),
    ("matapply_l5_bwd", "walk"), ("matapply_l5_bwd", "warp-per-token"),
    ("matapply_l5_fwd", "R kept"), ("matapply_l5_fwd", "R null"), ("matapply_l5_fwd", "walk"), ("matapply_l5_fwd", "warp-per-token"),
    ("pos_embed_bwd", "148-ranges"), ("pos_embed_bwd", "64-token-ranges"), ("pos_embed_bwd", "single-cta"),
    ("rowdiv_bwd", "critic"), ("rowdiv_bwd", "dff"), ("rowdiv_bwd", "qkv"), ("rowdiv_bwd", "walk"), ("rowdiv_bwd", "warp-per-token"),
    ("unfold_sym", "64-ctas-per-matrix"),
])


def test_regime_coverage(results):
    """The cases reach exactly these (kernel, regime) pairs: a change of a launcher that moves a case into another regime fails
    here instead of leaving the regime untested."""
    runs = {cid: results[cid] for cid in CASES}
    got = sorted(set().union(*(r.regimes for r in runs.values() if isinstance(r, Run))))
    failed = [cid for cid, r in runs.items() if not isinstance(r, Run)]
    assert got == REGIMES and not failed, (sorted(set(got) ^ set(REGIMES)), failed)
