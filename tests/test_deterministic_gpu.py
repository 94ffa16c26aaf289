"""Deterministic mode (sgrl_deterministic / SGRL_DETERMINISTIC=1): two runs of the same TD3 updates from the same state give
BIT-IDENTICAL parameters, like the reference's CPU autograd (src/agent.py:151,171), and still match the oracle step.  The
default mode sums split-K weight gradients and small cross-CTA reductions with fp32 atomics (order depends on timing)."""
import pytest
import torch

from sgrl_b200 import graph as G, morphologies as M, synth
from sgrl_b200._lib import lib
import parity
from test_agent_gpu import make_agent

pytestmark = pytest.mark.gpu


def run_updates(det, name, B, steps, use_graphs=True):
    prev = lib.sgrl_deterministic(1 if det else 0)
    try:
        ag, _, _ = make_agent(1)
        ag.use_graphs = use_graphs
        par = M.ALL[name]
        ag.change_morphology(G.build_graph(par, device="cuda"))
        gen = torch.Generator().manual_seed(5)
        losses = []
        for it in range(steps):
            b = {k: v.cuda() for k, v in synth.make_batch(B, len(par), seed=100 + it).items()}
            noise = (torch.randn(B, 3 * len(par), generator=gen) * 0.2).cuda()
            ld = ag.update(b, it, noise=noise)
            losses.append(ld["loss/critic_loss"].clone())
        torch.cuda.synchronize()
        arenas = [m.full_arena.detach().clone() for m in (ag.actor, ag.critic, ag.actor_target, ag.critic_target)]
        grads = [ag.critic.grad_arena().detach().clone(), ag.actor.grad_arena().detach().clone()]
        return arenas, grads, torch.stack(losses)
    finally:
        lib.sgrl_deterministic(prev)


@pytest.mark.parametrize("name,B,graphs", [("3d_humanoid_9_full", 256, True), ("3d_walker_7_full", 100, False)],
                         ids=["humanoid9-B256-graphs", "walker7-B100-eager"])
def test_two_runs_are_bit_identical(name, B, graphs):
    a1, g1, l1 = run_updates(True, name, B, 4, graphs)
    a2, g2, l2 = run_updates(True, name, B, 4, graphs)
    for x, y in zip(a1 + g1 + [l1], a2 + g2 + [l2]):
        assert torch.equal(x, y)


def test_deterministic_mode_matches_default_mode():
    """Same arithmetic, different summation order only: parameters after 4 updates agree to fp32 round-off."""
    ad, gd, ld = run_updates(True, "3d_humanoid_9_full", 256, 4)
    an, gn, ln = run_updates(False, "3d_humanoid_9_full", 256, 4)
    for x, y in zip(ad, an):
        assert parity.rel_err(x, y) < 1e-5
    for x, y in zip(gd, gn):
        assert parity.rel_err(x, y) < 1e-4
    assert parity.rel_err(ld, ln) < 1e-5
    report = [float((x != y).float().mean()) for x, y in zip(gd, gn)]
    print(f"  share of gradient elements that differ in the last bits between the two modes: critic {report[0]:.3f}, actor {report[1]:.3f}")


def test_mode_switch_is_reported():
    prev = lib.sgrl_deterministic(-1)
    assert lib.sgrl_deterministic(1) == prev
    assert lib.sgrl_deterministic(-1) == 1
    lib.sgrl_deterministic(prev)
    assert lib.sgrl_deterministic(-1) == prev

