"""Whole networks above the 592-graph switch of the attention forward (4 x 148 graphs: from there the second version,
attention_fwd_v2_kernel, runs; below it the first).  Every other parity test trains at B <= 256, below the switch.

* A twin-critic training pass (forward with the stash kept, backward with parameter, action and observation gradients)
  on 600 graphs is checked against the same graphs run as two 300-graph halves, which take the first version.
* All 23 CWHH morphologies x 26 samples (598 graphs, up to 15 limbs: NR = 16) packed into one batch against the
  per-morphology passes.
* The inference forward of 4 096 cheetah-14 envs (v2 NR = 16 without the probability store) against the fp64 oracle.
The batch sizes also put the head's K1 on a partial last token tile (T = 2 700, 5 400, 4 200, 8 400)."""
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import set_oracle as O
from sgrl_b200 import _lib, graph as G, morphologies as M, synth
from sgrl_b200.modules import make_packed_tables
import gpu_util
import parity
from test_gemm_gpu import TOL as GEMM_TOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=[1, 0], ids=["tcgen05", "simt"])
def mods(request):
    return gpu_util.make_modules(use_tc=request.param)


def attention_kernels(fn):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    return r, {e.name.split("(")[0].replace("void ", "").replace("sgrl::", "") for e in prof.events() if "attention_fwd" in e.name}


def one_signed_dout(T, seed):
    """A fixed per-token dL/dQ of one sign (uniform in [0.5, 1.5]).  The parameter gradients of the full batch and of the
    split batch differ only in the fp32 order of their sums over tokens; with random-sign dL/dQ the bias gradients (sums of
    dL/dQ) cancel to a small fraction of their terms, and a relative comparison would measure that cancellation instead."""
    return (torch.rand(2, T, 1, generator=torch.Generator().manual_seed(seed)) + 0.5).cuda()


def grad_tol(use_tc):
    """Bar of the per-tensor parameter-gradient comparison of a batch against the same batch split.  Q, dobs and dact of the
    two come out bit-identical, so the weight-gradient GEMMs see the same operands and differ only in how they reduce over
    the T tokens (one GEMM over T, or two over T/2 added; other split-K factors).  tests/test_gemm_gpu.py holds each such
    reduction within GEMM_TOL of fp64 (the tcgen05 accumulator truncates: 2e-5), so two of them may differ by twice that;
    1e-5 (the graph-vs-eager race test's scale) where that is larger.  Measured on a B200: 1.5e-5 worst on the tcgen05 path
    (cheetah-14, 8 400 tokens against two 4 200-token halves)."""
    return max(1e-5, 2 * GEMM_TOL[use_tc])


def train_pass(mod, tb, obs, act, dout, grads):
    """Twin-critic forward (stash kept) + backward: Q (2,T,1), dact (2,T,3), dobs (2,T,41); parameter gradients accumulate
    into `grads`."""
    q, stash = mod.forward_raw(tb, obs, act, keep=True, nb=2)
    dobs = torch.full((2, tb.T, 41), float("nan"), device="cuda")
    dact = mod.backward_raw(tb, stash, dout, 2, grads, True, dobs=dobs)
    torch.cuda.synchronize()
    return q, dact, dobs, stash


def per_graph_worst(got, ref, tok_graph, G):
    got, ref = got.double().reshape(got.shape[0], -1), ref.double().reshape(ref.shape[0], -1)
    num = torch.zeros(G, dtype=torch.float64, device="cuda").index_add_(0, tok_graph, ((got - ref) ** 2).sum(1))
    den = torch.zeros(G, dtype=torch.float64, device="cuda").index_add_(0, tok_graph, (ref ** 2).sum(1))
    return (num / den.clamp_min(1e-300)).sqrt().max().item()


def grad_errors(mod, got, ref):
    """[(name, rel err)] per live parameter tensor of every net of the arena."""
    out = []
    for z in range(mod._nb):
        for name, shape, off, live in _lib.param_table(mod._kind, mod._n_layers):
            if not live:
                continue
            n = 1
            for s in shape:
                n *= s
            a, b = got[z * mod._live + off: z * mod._live + off + n].double(), ref[z * mod._live + off: z * mod._live + off + n].double()
            if b.norm() == 0:
                out.append((f"{z}.{name}", a.norm().item()))
            else:
                out.append((f"{z}.{name}", ((a - b).norm() / b.norm()).item()))
    return out


@pytest.mark.parametrize("name,want", [("3d_humanoid_9_full", "attention_fwd_v2_kernel<12>"),
                                       ("3d_cheetah_14_full", "attention_fwd_v2_kernel<16>")])
def test_training_pass_above_switch_equals_two_halves(mods, name, want):
    _, critic, _, _ = mods
    par = M.ALL[name]
    N, B = len(par), 600
    g = G.build_graph(par, device="cuda")
    # data seed: one for which no relu unit of the full and split passes sits on its kink (the masks are compared below;
    # a unit within ~1e-7 of zero may land on either side under fp32 reassociation, DESIGN.md §2)
    b = gpu_util.to_cuda(synth.make_batch(B, N, seed=61))
    obs, act = b["obs"].view(-1, 41).contiguous(), b["action"].view(-1, 3).contiguous()
    tb = make_packed_tables([(g, B)], "cuda")
    halves = [make_packed_tables([(g, B // 2)], "cuda") for _ in range(2)]
    T, Th = tb.T, halves[0].T
    dout = one_signed_dout(T, 62)

    grads_full = torch.zeros(critic._nb * critic._live, device="cuda")
    (q, dact, dobs, stash), k_full = attention_kernels(lambda: train_pass(critic, tb, obs, act, dout, grads_full))
    assert k_full == {want}, k_full
    grads_split = torch.zeros_like(grads_full)
    parts = []
    for i, th in enumerate(halves):
        sl = slice(i * Th, (i + 1) * Th)
        r, k_half = attention_kernels(lambda: train_pass(critic, th, obs[sl].contiguous(), act[sl].contiguous(),
                                                         dout[:, sl].contiguous(), grads_split))
        assert k_half == {"attention_fwd_kernel"}, k_half
        parts.append(r)

    for z in range(2):
        full_mk = gpu_util.relu_masks(critic, stash, tb, 2, z)
        half_mk = [gpu_util.relu_masks(critic, r[3], halves[i], 2, z) for i, r in enumerate(parts)]
        for key, m in full_mk.items():
            assert torch.equal(m, torch.cat([h[key] for h in half_mk])), f"relu mask {key} of net {z} differs"

    q_s = torch.cat([r[0] for r in parts], 1)
    dact_s = torch.cat([r[1] for r in parts], 1)
    dobs_s = torch.cat([r[2] for r in parts], 1)
    dq = (q - q_s).abs().max().item()
    print(f"\n{name} B={B}: Q full vs halves max |diff| {dq:.2e} (bitwise: {torch.equal(q, q_s)})")
    assert dq <= 1e-6 * q_s.abs().max().item()
    tok_graph = torch.arange(B, device="cuda").repeat_interleave(N)
    for z in range(2):
        e_obs = per_graph_worst(dobs[z], dobs_s[z], tok_graph, B)
        e_act = per_graph_worst(dact[z], dact_s[z], tok_graph, B)
        print(f"  net {z}: worst graph dobs {e_obs:.2e}, dact {e_act:.2e}")
        assert e_obs <= 1e-5 and e_act <= 1e-5
    ge = grad_errors(critic, grads_full, grads_split)
    print(f"  parameter gradients: worst tensor {max(ge, key=lambda x: x[1])}")
    bad = [(k, e) for k, e in ge if e > grad_tol(critic.use_tc)]
    assert not bad, bad[:8]


def test_packed_cwhh_above_switch_equals_per_morphology(mods):
    """23 morphologies x 26 samples = 598 graphs of up to 15 limbs in one batch: v2 NR = 16 for the forward with and without
    the probability store.  Forwards equal the per-morphology forwards, a packed backward the sum of the per-morphology ones."""
    actor, critic, _, _ = mods
    names = sorted(M.CWHH)
    assert len(names) == 23
    B = 26
    graphs = [G.build_graph(M.ALL[n], device="cuda") for n in names]
    batches = [gpu_util.to_cuda(synth.make_batch(B, len(M.ALL[n]), seed=70 + i)) for i, n in enumerate(names)]
    tb = make_packed_tables([(g, B) for g in graphs], "cuda")
    assert tb.G == 598 and tb.nmax > 12
    obs = torch.cat([b["obs"].view(-1, 41) for b in batches]).contiguous()
    act = torch.cat([b["action"].view(-1, 3) for b in batches]).contiguous()
    dq = one_signed_dout(tb.T, 71)
    with torch.no_grad():
        (pi, _), k_a = attention_kernels(lambda: actor.forward_raw(tb, obs, None, keep=False))
        assert k_a == {"attention_fwd_v2_kernel<16>"}, k_a
    grads_p = torch.zeros(critic._nb * critic._live, device="cuda")
    (q, dact, dobs, _), k_c = attention_kernels(lambda: train_pass(critic, tb, obs, act, dq, grads_p))
    assert k_c == {"attention_fwd_v2_kernel<16>"}, k_c
    grads_m = torch.zeros_like(grads_p)
    worst = {"pi": 0.0, "q": 0.0, "dobs": 0.0, "dact": 0.0}
    for (t0, t1, _, _, n), g, b in zip(tb.parts, graphs, batches):
        one = make_packed_tables([(g, B)], "cuda")
        o_obs, o_act = b["obs"].view(-1, 41).contiguous(), b["action"].view(-1, 3).contiguous()
        with torch.no_grad():
            pi1, _ = actor.forward_raw(one, o_obs, None, keep=False)
        q1, dact1, dobs1, _ = train_pass(critic, one, o_obs, o_act, dq[:, t0:t1].contiguous(), grads_m)
        for key, a, r in (("pi", pi[:, t0:t1], pi1), ("q", q[:, t0:t1], q1), ("dobs", dobs[:, t0:t1], dobs1),
                          ("dact", dact[:, t0:t1], dact1)):
            worst[key] = max(worst[key], parity.rel_err(a, r))
    print(f"\nCWHH x {B} packed vs per morphology: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    # the per-morphology batches (78..390 tokens) run other GEMM tilings and variants than the packed 5 564-token batch,
    # and the attention bias sums in another contraction (v1 vs v2): fp32 reassociation through three layers, 2.7e-6 at most
    # measured on a B200, under the 1e-5 of the packed-vs-per-morphology forward test
    assert worst["pi"] <= 1e-5 and worst["q"] <= 1e-5, worst
    assert worst["dobs"] <= 1e-5 and worst["dact"] <= 1e-5, worst
    ge = grad_errors(critic, grads_p, grads_m)
    print(f"  parameter gradients: worst tensor {max(ge, key=lambda x: x[1])}")
    bad = [(k, e) for k, e in ge if e > grad_tol(critic.use_tc)]
    assert not bad, bad[:8]


def test_inference_v2_nr16_forward_4096_cheetahs(mods):
    """The rollout's actor forward of 4 096 cheetah-14 envs (57 344 tokens; persistent GEMMs; attention v2 NR = 16 without
    the probability store) against the fp64 oracle at the 1e-4 bar, and invariant to a rotation about gravity at 1e-5."""
    actor, _, pa, _ = mods
    par = M.ALL["3d_cheetah_14_full"]
    g = G.build_graph(par, device="cuda")
    actor.change_morphology(g)
    obs = synth.make_obs(4096, len(par), seed=81).cuda()
    with torch.no_grad():
        got, k = attention_kernels(lambda: actor(obs))
        assert k == {"attention_fwd_v2_kernel<16>"}, k
        p64 = {kk: v.cuda().double() for kk, v in pa.items()}
        g64 = dict(g, relation=g["relation"].double())
        want = O.actor_forward(p64, obs.double(), g64)
    err = parity.rel_err(got, want)
    print(f"\ncheetah-14 x 4096 forward: rel err {err:.2e}")
    assert err < parity.RTOL
    rot = synth.rotate_about_gravity(obs.cpu(), len(par), 0.7).cuda()
    with torch.no_grad():
        err_rot = parity.rel_err(actor(rot), got)
    assert err_rot < parity.RTOL_ROT
