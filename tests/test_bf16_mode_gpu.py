"""BF16-input mode (use_tc = 2; north_star: "fp32 accumulate, bf16 inputs stated separately").  Both operands of every
tcgen05 projection are rounded to bf16 (RN-even) in the operand path and multiplied in ONE tensor-core pass with fp32
accumulation — numerically a bf16 x bf16 -> f32 MMA.  Never the default and never the headline number.

* the GEMM itself is exact for that definition: equal to an fp64 product of the bf16-rounded operands up to fp32
  accumulation error, for the three contraction forms of the hot path;
* the networks' measured accuracy against the fp64 oracle is recorded (printed) and bounded: actions, Q, gradients and the
  rotation-about-gravity invariance are at bf16 level (1e-3..1e-2), NOT at the fp32 parity bar — which is why the mode is
  reported separately.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import set_oracle as O
from sgrl_b200 import graph as G, morphologies as M, synth
import gpu_util
import parity
from test_backward_gpu import grad_report, oracle_grads
from test_gemm_gpu import rel, run_gemm

pytestmark = pytest.mark.gpu


def bf(x):
    return x.bfloat16().double()


@pytest.mark.parametrize("M_,N,K", [(2304, 768, 256), (300, 256, 1024), (1000, 128, 544)])
def test_gemm_forward_is_a_bf16_input_product(M_, N, K):
    g = torch.Generator(device="cuda").manual_seed(N)
    X, W = torch.randn(M_, K, device="cuda", generator=g), torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    Y = torch.empty(M_, N, device="cuda")
    run_gemm(X, K, 0, W, K, 0, Y, N, M_, N, K, bias=b, use_tc=2)
    assert rel(Y, bf(X) @ bf(W).T + b.double()) < 5e-6
    assert rel(Y, X.double() @ W.double().T + b.double()) > 5e-4            # and it is NOT the fp32-parity product


def test_gemm_data_and_weight_gradient_forms():
    g = torch.Generator(device="cuda").manual_seed(1)
    T, Nw, Kw = 2304, 768, 256
    dY, W, X = torch.randn(T, Nw, device="cuda", generator=g), torch.randn(Nw, Kw, device="cuda", generator=g), torch.randn(T, Kw, device="cuda", generator=g)
    dX = torch.zeros(T, Kw, device="cuda")
    run_gemm(dY, Nw, 0, W, Kw, 1, dX, Kw, T, Kw, Nw, use_tc=2)                              # dX = dY W
    assert rel(dX, bf(dY) @ bf(W)) < 5e-6
    dW = torch.zeros(Nw, Kw, device="cuda")
    run_gemm(dY, Nw, 1, X, Kw, 1, dW, Kw, Nw, Kw, T, acc=1, splitk=4, use_tc=2)             # dW += dY^T X
    assert rel(dW, bf(dY).T @ bf(X)) < 5e-6


def test_network_accuracy_in_bf16_input_mode_is_recorded_and_bounded(capsys):
    actor, critic, pa, pc = gpu_util.make_modules(use_tc=2)
    par = M.ALL["3d_humanoid_9_full"]
    g = G.build_graph(par, device="cuda")
    actor.change_morphology(g); critic.change_morphology(g)
    b = gpu_util.to_cuda(synth.make_batch(256, len(par), seed=1))
    g64 = dict(g); g64["relation"] = g["relation"].double()
    pa64, pc64 = {k: v.cuda().double() for k, v in pa.items()}, {k: v.cuda().double() for k, v in pc.items()}
    with torch.no_grad():
        a = actor(b["obs"])
        q1, q2 = critic(b["obs"], b["action"])
        a_ref = O.actor_forward(pa64, b["obs"].double(), g64)
        q1_ref, q2_ref = O.critic_forward(pc64, b["obs"].double(), b["action"].double(), g64)
        rot = synth.rotate_about_gravity(b["obs"], len(par), 0.7)
        e_rot_a = parity.rel_err(actor(rot), a)
        e_rot_q = parity.rel_err(critic(rot, b["action"])[0], q1)
    e_a, e_q = parity.rel_err(a, a_ref), max(parity.rel_err(q1, q1_ref), parity.rel_err(q2, q2_ref))
    critic.zero_grad(set_to_none=True)
    o1, o2 = critic(b["obs"], b["action"])
    tgt = b["reward"].expand_as(o1)
    (F.mse_loss(o1, tgt) + F.mse_loss(o2, tgt)).backward()
    got = {k: p.grad for k, p in critic.named_parameters()}

    def lf(p):
        r1, r2 = O.critic_forward(p, b["obs"].double(), b["action"].double(), g64)
        t = b["reward"].double().expand_as(r1)
        return F.mse_loss(r1, t) + F.mse_loss(r2, t)
    _, want = oracle_grads(pc, lf)
    bad, glob = grad_report(got, want, rtol=1.0)
    worst = max((parity.rel_err(got[k], w) for k, w in want.items() if w is not None and not k.endswith("rel_encoder.bias") and float(w.norm()) > 1e-4 * float(
        torch.sqrt(sum((v.double() ** 2).sum() for v in want.values() if v is not None)))), default=0.0)
    with capsys.disabled():
        print(f"\nBF16-input mode, humanoid-9 B=256 vs the fp64 oracle: actions {e_a:.2e}, Q {e_q:.2e}, critic gradients global {glob:.2e} "
              f"(worst tensor {worst:.2e}); rotation about gravity: actions {e_rot_a:.2e}, Q {e_rot_q:.2e}")
    assert e_a < 5e-2 and e_q < 5e-2 and glob < 1e-1 and e_rot_a < 5e-2 and e_rot_q < 5e-2
    assert e_a > parity.RTOL or e_q > parity.RTOL        # a reduced-precision mode: it must not be mistaken for the parity path


def test_persistent_kernels_in_bf16_input_mode():
    """At rollout sizes the BF16-input mode runs its projections in the persistent tcgen05 kernels too (one MMA pass per
    k-block, the weights' lo tile is not even loaded).  The per-tile kernels run the same forward when it keeps its activations
    for a backward (the planner gives persistent kernels only to passes that keep nothing).  The short-K projections
    accumulate in the same order as the per-tile kernels (bit-identical); the K = 544 Gram projection sums 17 k-blocks on one
    accumulator instead of two, and a 1e-7 difference in an activation that sits on a bf16 rounding boundary becomes a bf16 ulp
    (4e-3) in the next projection's operand — so the two schedules agree at the mode's own noise level, and both are equally
    far from the fp64 oracle."""
    from test_agent_gpu import make_agent
    ag, pa, _ = make_agent(2)
    par = M.ALL["3d_walker_7_full"]
    g = G.build_graph(par, device="cuda")
    ag.change_morphology(g)
    obs = synth.make_obs(8192, len(par), seed=21).cuda()              # 57 344 tokens: 448 row tiles
    with torch.no_grad():
        got = ag.actor(obs).clone()
        want, _ = ag.actor.forward_raw(ag.actor._tables(obs.shape[0]), obs, None, keep=True, nb=1)
        want = want[0].reshape(got.shape)
        ref = O.actor_forward({k: v.cuda() for k, v in pa.items()}, obs, g)
    e_pt, e_p, e_t = parity.rel_err(got, want), parity.rel_err(got, ref), parity.rel_err(want, ref)
    print(f"  BF16-input mode at 57k tokens: persistent vs per-tile {e_pt:.2e}; vs the oracle: persistent {e_p:.2e}, per-tile {e_t:.2e}")
    assert e_pt < 5e-3
    assert e_p < 2e-2 and e_t < 2e-2 and e_p < 1.5 * e_t + 1e-3
