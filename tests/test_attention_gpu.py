"""K2, the attention core, through the C ABI (sgrl_attention_fwd / sgrl_attention_bwd) against the fp64 references of
tests/kernel_ref.py, in every launch regime the update and the rollout reach:

  attention_fwd_kernel          G < 4 * 148 graphs (grid-stride over graphs above 2 CTAs/SM x 148 for 9..16-limb graphs)
  attention_fwd_v2_kernel<12>   G >= 592, largest graph <= 12 limbs
  attention_fwd_v2_kernel<16>   G >= 592, largest graph 13..16 limbs (or the hint 0 = unknown)
  attention_bwd_kernel          one CTA/SM for 16-limb graphs: grid-stride above 148 graphs; one CTA in deterministic
                                mode without scratch

Errors are taken per graph (the worst graph of the batch, not the batch norm: one wrong graph out of thousands moves a
batch norm by little), outputs are NaN-prefilled with pad rows past T that must stay untouched, and each regime case
asserts from a torch.profiler trace which kernel ran, so that a change of the 592 threshold cannot make it vacuous."""

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import kernel_ref as R

pytestmark = pytest.mark.gpu

PAD = 5                  # sentinel rows past T in every output buffer
V2_MIN = 4 * 148         # the graph count from which the forward runs the second version
TOL_GRAPH = 1e-5         # worst graph, relative (o, og, dqkv, dvgp)
TOL_P = 1e-6             # probabilities, absolute
TOL_BATCH = 2e-6         # whole batch, relative


def _lib():
    from sgrl_b200 import _lib
    return _lib


def make_case(sizes, seed, bias="ragged", score_scale=1.0):
    """Packed inputs of graphs with `sizes` limbs.  q, k entries of std 128^-1/4 give scores of order 1 (score_scale
    multiplies them); bias: None, "ragged" (one (n,n,3) table per graph at rel_off[g]) or "null" (rel_off NULL: every
    graph reads the table at offset 0)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    sizes = torch.as_tensor(sizes, dtype=torch.int64)
    cu = torch.zeros(len(sizes) + 1, dtype=torch.int32)
    cu[1:] = torch.cumsum(sizes, 0)
    T = int(cu[-1])
    qkv = torch.randn(T, 768, device="cuda", generator=g)
    qkv[:, :512] *= 128 ** -0.25 * score_scale ** 0.5
    c = dict(G=len(sizes), T=T, sizes=sizes, cu=cu.cuda(), qkv=qkv,
             vgp=torch.randn(T, 756, device="cuda", generator=g), gd=torch.randn(T, 6, device="cuda", generator=g),
             rw=None, rb=None, rel_off=None, relation=None, nmax=int(sizes.max()))
    if bias is not None:
        c["rw"] = torch.randn(2, 3, device="cuda", generator=g) * 0.5
        c["rb"] = torch.randn(2, device="cuda", generator=g) * 0.5
        if bias == "ragged":
            nn3 = sizes * sizes * 3
            off = torch.zeros(len(sizes), dtype=torch.int32)
            off[1:] = torch.cumsum(nn3, 0)[:-1].to(torch.int32)
            c["rel_off"] = off.cuda()
            c["relation"] = torch.rand(int(nn3.sum()), device="cuda", generator=g)
        else:
            c["relation"] = torch.rand(16 * 16 * 3, device="cuda", generator=g)
    c["tok_graph"] = torch.repeat_interleave(torch.arange(len(sizes)), sizes).cuda()
    return c


def ragged_sizes(G, lo, hi, seed, must=()):
    """G graph sizes drawn uniformly from lo..hi in random order (large graphs followed by small ones in the same CTA),
    with the sizes in `must` placed at random positions."""
    g = torch.Generator().manual_seed(seed)
    s = torch.randint(lo, hi + 1, (G,), generator=g)
    pos = torch.randperm(G, generator=g)[:len(must)]
    s[pos] = torch.tensor(must, dtype=torch.int64)[:len(pos)]
    return s


def sentinel(T, *shape):
    return torch.full((T + PAD, *shape), float("nan"), device="cuda")


def run_fwd(c, max_limbs=None, store_p=True, kernels=None):
    """o, og, p (p None without the store) of the kernel, or with kernels=[] also the names of the kernels it launched."""
    L = _lib()
    T = c["T"]
    o, og = sentinel(T, 256), sentinel(T, 768)
    p = sentinel(T, 32) if store_p else None
    ml = c["nmax"] if max_limbs is None else max_limbs
    call = lambda: L.check(L.lib.sgrl_attention_fwd(L.ptr(c["qkv"]), L.ptr(c["vgp"]), L.ptr(c["gd"]), L.ptr(c["rw"]), L.ptr(c["rb"]),
                                                    L.ptr(c["cu"]), L.ptr(c["rel_off"]), L.ptr(c["relation"]), c["G"], ml,
                                                    L.ptr(o), L.ptr(og), L.ptr(p), L.stream()), "sgrl_attention_fwd")
    if kernels is None:
        call()
    else:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        kernels += [e.name for e in prof.events() if "attention" in e.name]
    torch.cuda.synchronize()
    for buf in (o, og) + ((p,) if store_p else ()):
        assert torch.isnan(buf[T:]).all(), "a pad row past T was written"
        assert torch.isfinite(buf[:T]).all(), "a row < T was left unwritten or is not finite"
    return o[:T], og[:T], (p[:T] if store_p else None)


def run_bwd(c, p, d_o, d_og, max_limbs=None, drel_prefill=0.25):
    L = _lib()
    T = c["T"]
    dqkv, dvgp = sentinel(T, 768), sentinel(T, 756)
    drel = None if c["rw"] is None else torch.full((2, 3), drel_prefill, device="cuda")
    ml = c["nmax"] if max_limbs is None else max_limbs
    L.check(L.lib.sgrl_attention_bwd(L.ptr(c["qkv"]), L.ptr(c["vgp"]), L.ptr(c["gd"]), L.ptr(p), L.ptr(d_o), L.ptr(d_og),
                                      L.ptr(c["cu"]), L.ptr(c["rel_off"]), L.ptr(c["relation"]), c["G"], ml,
                                      L.ptr(dqkv), L.ptr(dvgp), L.ptr(drel), L.stream()), "sgrl_attention_bwd")
    torch.cuda.synchronize()
    for buf in (dqkv, dvgp):
        assert torch.isnan(buf[T:]).all(), "a pad row past T was written"
        assert torch.isfinite(buf[:T]).all(), "a row < T was left unwritten or is not finite"
    return dqkv[:T], dvgp[:T], drel


def ref_fwd(c):
    return R.attention_fwd_ref(c["qkv"], c["vgp"], c["gd"], c["rw"], c["rb"], c["cu"], c["rel_off"], c["relation"])


def ref_bwd(c, d_o, d_og):
    return R.attention_bwd_ref(c["qkv"], c["vgp"], c["gd"], c["rw"], c["rb"], c["cu"], c["rel_off"], c["relation"], d_o, d_og)


def graph_err(got, ref, c):
    """(worst per-graph relative error, graph index, whole-batch relative error)."""
    got, ref = got.double().reshape(c["T"], -1), ref.reshape(c["T"], -1)
    num = torch.zeros(c["G"], dtype=torch.float64, device="cuda").index_add_(0, c["tok_graph"], ((got - ref) ** 2).sum(1))
    den = torch.zeros(c["G"], dtype=torch.float64, device="cuda").index_add_(0, c["tok_graph"], (ref ** 2).sum(1))
    e = (num / den.clamp_min(1e-300)).sqrt()
    worst = int(torch.argmax(e))
    return e[worst].item(), worst, ((got - ref).norm() / ref.norm()).item()


def check_fwd(c, o, og, p):
    ro, rog, rp = ref_fwd(c)
    errs = {}
    for name, got, ref in (("o", o, ro), ("og", og, rog)):
        worst, gi, batch = graph_err(got, ref, c)
        assert worst <= TOL_GRAPH, f"{name}: graph {gi} ({int(c['sizes'][gi])} limbs) rel err {worst:.2e}"
        assert batch <= TOL_BATCH, f"{name}: batch rel err {batch:.2e}"
        errs[name] = worst
    if p is not None:
        p = p.view(c["T"], 2, 16)
        dp = (p.double() - rp).abs()
        errs["p"] = dp.max().item()
        assert errs["p"] <= TOL_P, f"p: max abs err {errs['p']:.2e} at token {int(dp.amax((1, 2)).argmax())}"
        n_tok = c["sizes"].cuda()[c["tok_graph"]]
        beyond = torch.arange(16, device="cuda")[None, None, :] >= n_tok[:, None, None]
        assert torch.all(p[beyond.expand_as(p)] == 0.0), "p[t, h, j] must be exactly 0 for j >= n"
    return errs


def check_bwd(c, p, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    d_o = torch.randn(c["T"], 256, device="cuda", generator=g)
    d_og = torch.randn(c["T"], 768, device="cuda", generator=g)
    dqkv, dvgp, drel = run_bwd(c, p, d_o, d_og)
    rq, rv, rw = ref_bwd(c, d_o, d_og)
    errs = {}
    for name, got, ref in (("dqkv", dqkv, rq), ("dvgp", dvgp, rv)):
        worst, gi, batch = graph_err(got, ref, c)
        assert worst <= TOL_GRAPH, f"{name}: graph {gi} ({int(c['sizes'][gi])} limbs) rel err {worst:.2e}"
        assert batch <= TOL_BATCH, f"{name}: batch rel err {batch:.2e}"
        errs[name] = worst
    if drel is not None:       # accumulates into what was there; exactly 0 for one-limb graphs (dS = 0), hence the clamp
        errs["drel_w"] = ((drel.double() - 0.25 - rw).norm() / rw.norm().clamp_min(1e-30)).item()
        assert errs["drel_w"] <= TOL_GRAPH, errs
    return errs


def expected_fwd_kernel(G, nmax_hint):
    if G < V2_MIN:
        return "attention_fwd_kernel("
    nr = nmax_hint if 2 <= nmax_hint <= 16 else 16
    return "attention_fwd_v2_kernel<12>" if nr <= 12 else "attention_fwd_v2_kernel<16>"


def assert_kernel(names, want):
    assert names and all(want in n for n in names), f"expected {want}, the trace shows {names}"


# ---------------------------------------------------------------------------------------------------------------- regimes
REGIMES = [1, 148, 149, 591, 592, 2400, 6000]


@pytest.mark.parametrize("wide", [False, True], ids=["max12", "max16"])
@pytest.mark.parametrize("G", REGIMES)
def test_regime_forward_backward(G, wide):
    """Ragged graphs with a per-graph relation table: forward (P stored) and backward on the kernel's own P."""
    must = (16, 13, 15, 14) if wide else (12, 2, 11)
    sizes = ragged_sizes(G, 1, 16 if wide else 12, seed=G * 2 + wide, must=must)
    c = make_case(sizes, seed=G + 17 * wide)
    names = []
    o, og, p = run_fwd(c, kernels=names)
    want = expected_fwd_kernel(G, c["nmax"])
    assert_kernel([n for n in names if "fwd" in n], want)
    errs = check_fwd(c, o, og, p)
    errs.update(check_bwd(c, p, seed=G))
    print(f"\nK2 regime G={G} nmax={c['nmax']} kernel={want.rstrip('(')} " + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))


@pytest.mark.parametrize("G", [37, 700])
@pytest.mark.parametrize("n", list(range(1, 17)))
def test_uniform_limb_count(n, G):
    """Each n = 1..16 as a uniform batch (n = 1: the softmax of one key is 1; n = 16: a full tile), both versions."""
    c = make_case([n] * G, seed=100 + n)
    names = []
    o, og, p = run_fwd(c, kernels=names)
    assert_kernel([x for x in names if "fwd" in x], expected_fwd_kernel(G, n))
    check_fwd(c, o, og, p)
    if n == 1:
        assert torch.all(p.view(-1, 2, 16)[:, :, 0] == 1.0)
    check_bwd(c, p, seed=n)


@pytest.mark.parametrize("bias", [None, "ragged", "null"])
@pytest.mark.parametrize("G", [300, 2400])
def test_relation_bias_variants(bias, G):
    c = make_case(ragged_sizes(G, 2, 16, seed=5, must=(16,)), seed=6, bias=bias)
    o, og, p = run_fwd(c)
    check_fwd(c, o, og, p)
    check_bwd(c, p, seed=7)


# ------------------------------------------------------------------------------------------------------- max_limbs hint
def test_max_limbs_hint():
    """The hint sizes the staging and picks NR: exact, 0 (unknown -> 16) and larger than needed all compute the same.
    12-limb graphs with hint 12 run NR = 12 and with hint 13 NR = 16; 9-limb graphs with hint 9 vs 0 likewise.  The
    accumulator rows only change which registers hold the sums, not their arithmetic: the results are bit-identical."""
    for n, hints in ((12, (12, 13, 0, 16)), (9, (9, 0, 14))):
        c = make_case(ragged_sizes(700, 1, n, seed=n, must=(n,)), seed=n, bias=None)
        outs = []
        for h in hints:
            names = []
            outs.append(run_fwd(c, max_limbs=h, kernels=names))
            assert_kernel(names, expected_fwd_kernel(c["G"], h))
        check_fwd(c, *outs[0])
        for other in outs[1:]:
            for a, b in zip(outs[0], other):
                assert torch.equal(a, b)
        # v1 with a hint larger than needed
        c1 = make_case(ragged_sizes(200, 1, n, seed=n + 1, must=(n,)), seed=n + 1)
        for h in (n, 0, 16):
            check_fwd(c1, *run_fwd(c1, max_limbs=h))


# ------------------------------------------------------------------------------------------------------------- bitwise
@pytest.mark.parametrize("bias", [None, "ragged"])
def test_v1_v2_same_arithmetic(bias):
    """v1 and v2 accumulate in the same order: graphs 0..590 launched as 591 graphs (v1) and with one more graph (v2)
    give bit-identical o, og and p without a bias.  With the bias, `wr . rr + br` is a short expression whose fp
    contraction into FMAs may differ between the two kernels: there the outputs agree to a few ulp of fp32."""
    sizes = ragged_sizes(V2_MIN, 1, 16, seed=11, must=(16, 13))
    full = make_case(sizes, seed=12, bias=bias)
    part = dict(full, G=V2_MIN - 1, T=int(full["cu"][V2_MIN - 1]), sizes=sizes[:-1], cu=full["cu"][:V2_MIN],
                tok_graph=full["tok_graph"][:int(full["cu"][V2_MIN - 1])])
    n1, n2 = [], []
    a = run_fwd(part, kernels=n1)
    b = run_fwd(full, kernels=n2)
    assert_kernel(n1, "attention_fwd_kernel(")
    assert_kernel(n2, "attention_fwd_v2_kernel<16>")
    T = part["T"]
    for x, y in zip(a, b):
        if bias is None:
            assert torch.equal(x, y[:T])
        else:
            assert (x - y[:T]).abs().max().item() <= 4 * torch.finfo(torch.float32).eps * y[:T].abs().max().item()


@pytest.mark.parametrize("G", [300, 2400])
def test_inference_pass_without_p(G):
    """p = NULL (the rollout's inference pass): the same o and og, bit for bit, as the launch that stores P."""
    c = make_case(ragged_sizes(G, 2, 16, seed=21, must=(16,)), seed=22)
    o, og, _ = run_fwd(c)
    names = []
    o2, og2, none = run_fwd(c, store_p=False, kernels=names)
    assert none is None
    assert_kernel(names, expected_fwd_kernel(G, c["nmax"]))
    assert torch.equal(o, o2) and torch.equal(og, og2)


def test_large_logits():
    """Scores of order +-100: the max subtraction keeps every output finite and P within 1e-4 of fp64 per element."""
    for G in (300, 2400):
        c = make_case(ragged_sizes(G, 1, 16, seed=31, must=(16,)), seed=32, score_scale=100.0)
        o, og, p = run_fwd(c)
        _, _, rp = ref_fwd(c)
        p = p.view(-1, 2, 16)
        assert (p.double() - rp).abs().max().item() <= 1e-4
        assert (p.double().sum(-1) - 1).abs().max().item() <= 1e-6
        assert (rp.amax(-1) > 0.9).float().mean().item() > 0.5, "the scores are not large enough to test the max subtraction"


# -------------------------------------------------------------------------------------------------- deterministic mode
def test_backward_deterministic_one_cta():
    """sgrl_deterministic(1) with drel_w and no scratch: one CTA walks every graph.  Two runs are bit-identical; dqkv and
    dvgp equal the default mode's bit for bit (same per-graph arithmetic, other grid).  drel_w sums the same 600 graphs'
    terms in another order (one CTA instead of fp32 atomics from many): both agree with fp64 to 1e-5 and with each other
    to 5e-6 (1.2e-6 measured on a B200: the per-graph terms cancel, ||sum|| is below the sum of their norms)."""
    L = _lib()
    c = make_case(ragged_sizes(600, 1, 16, seed=41, must=(16,)), seed=42)
    o, og, p = run_fwd(c)
    g = torch.Generator(device="cuda").manual_seed(43)
    d_o = torch.randn(c["T"], 256, device="cuda", generator=g)
    d_og = torch.randn(c["T"], 768, device="cuda", generator=g)
    base = run_bwd(c, p, d_o, d_og)
    prev = L.lib.sgrl_deterministic(1)
    try:
        r1 = run_bwd(c, p, d_o, d_og)
        r2 = run_bwd(c, p, d_o, d_og)
    finally:
        L.lib.sgrl_deterministic(prev)
    for x, y in zip(r1, r2):
        assert torch.equal(x, y)
    assert torch.equal(r1[0], base[0]) and torch.equal(r1[1], base[1])
    assert ((r1[2] - base[2]).norm() / (base[2] - 0.25).norm()).item() <= 5e-6
    _, _, rw = ref_bwd(c, d_o, d_og)
    for r in (r1, base):
        assert ((r[2].double() - 0.25 - rw).norm() / rw.norm()).item() <= TOL_GRAPH
