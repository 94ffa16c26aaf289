"""CPU pins of the observation gradient the GPU tests compare against: the oracle's fp64 d/d(state) equals the unmodified
reference modules' (when the reference is on this machine), and it rotates with the limb vectors about gravity."""
import pytest
import torch

from oracle import ref_loader, set_oracle as O
from sgrl_b200 import graph as G, morphologies as M, synth
import parity


@pytest.mark.skipif(ref_loader.find_reference() is None, reason="reference not on this machine")
def test_oracle_state_gradient_against_live_reference():
    ref = ref_loader.load_reference()
    torch.manual_seed(0)
    ag = ref.agent.Agent(ref_loader.default_args())
    par = M.ALL["3d_humanoid_8_left_knee"]
    g = ref.utils.getGraphDict(par, ["pre", "inlcrs", "postlcrs"], device=torch.device("cpu"))
    ag.change_morphology(g)
    sd = ag.state_dict()
    pa = {k[len("actor."):]: v.double() for k, v in sd.items() if k.startswith("actor.")}
    pc = {k[len("critic."):]: v.double() for k, v in sd.items() if k.startswith("critic.")}
    b = synth.make_batch(6, len(par), seed=9)
    c = torch.randn(b["action"].shape, generator=torch.Generator().manual_seed(2))
    g64 = dict(g); g64["relation"] = g["relation"].double()

    s = b["obs"].clone().requires_grad_(True)
    q1, q2 = ag.critic(s, b["action"])
    (q1.sum() + 2.0 * q2.sum()).backward()
    s64 = b["obs"].double().requires_grad_(True)
    o1, o2 = O.critic_forward(pc, s64, b["action"].double(), g64)
    (o1.sum() + 2.0 * o2.sum()).backward()
    assert parity.rel_err(s.grad, s64.grad) < parity.RTOL

    s = b["obs"].clone().requires_grad_(True)
    (ag.actor(s) * c).sum().backward()
    s64 = b["obs"].double().requires_grad_(True)
    (O.actor_forward(pa, s64, g64) * c.double()).sum().backward()
    assert parity.rel_err(s.grad, s64.grad) < parity.RTOL


def test_oracle_state_gradient_rotates_with_the_limb_vectors():
    """an invariant loss has a gradient whose 8 limb vectors rotate with the input and whose 17 scalars do not change"""
    par = M.ALL["3d_hopper_3_shin"]
    n = len(par)
    g = G.build_graph(par)
    g["relation"] = g["relation"].double()
    pc = {k: v.double() for k, v in O.synth_params("critic", parity.WEIGHT_SEED + 1).items()}
    b = synth.make_batch(3, n, seed=2)
    angle = 0.7

    def grad_at(obs):
        s = obs.double().clone().requires_grad_(True)
        q = O.transformer_model(pc, torch.cat([s.view(3, n, 41), b["action"].double().view(3, n, 3)], 2), g)
        (q ** 2).sum().backward()
        return s.grad
    g0 = grad_at(b["obs"])
    gr = grad_at(synth.rotate_about_gravity(b["obs"].double(), n, angle))
    assert parity.rel_err(gr, synth.rotate_about_gravity(g0, n, angle)) < 1e-10
    assert parity.rel_err(gr, g0) > 1e-2
