"""Agent.update / select_action on the GPU vs the TD3 oracle (torch Adam + clip_grad_norm_)
and vs the reference's recorded update steps."""
import numpy as np
import pytest
import torch

from oracle import ref_loader, set_oracle as O
from sgrl_b200 import graph as G, morphologies as M, synth
import parity

pytestmark = pytest.mark.gpu


def make_agent(use_tc=1):
    from sgrl_b200.agent import Agent
    ag = Agent(ref_loader.default_args())
    a = O.synth_params("actor", parity.WEIGHT_SEED)
    c1 = O.synth_params("critic", parity.WEIGHT_SEED + 1)
    c2 = O.synth_params("critic", parity.WEIGHT_SEED + 2)
    sd = {}
    for pre in ("actor.actor.", "actor_target.actor."):
        sd.update({pre + k: v for k, v in a.items()})
    for pre in ("critic.", "critic_target."):
        sd.update({pre + "critic1." + k: v for k, v in c1.items()})
        sd.update({pre + "critic2." + k: v for k, v in c2.items()})
    ag.load_state_dict(sd)
    for m in (ag.actor, ag.actor_target, ag.critic, ag.critic_target):
        m.use_tc = use_tc
    pa = {"actor." + k: v for k, v in a.items()}
    pc = {"critic1." + k: v for k, v in c1.items()}
    pc.update({"critic2." + k: v for k, v in c2.items()})
    return ag, pa, pc


def agent_state(ag):
    return {k: v.detach().clone() for k, v in ag.state_dict().items()}


def test_state_dict_has_reference_keys():
    ag, _, _ = make_agent()
    gold = parity.load_golden()
    assert list(ag.state_dict().keys()) == [str(s) for s in gold["state_names"]]
    assert len(ag.state_dict()) == 818


@pytest.mark.parametrize("use_tc", [1, 0], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("name,B", [parity.CASES[1], parity.CASES[3]])
def test_update_matches_reference_golden(name, B, use_tc):
    gold = parity.load_golden()
    ag, _, _ = make_agent(use_tc)
    g = parity.golden_graph(gold, name, M.ALL[name], device="cuda")
    b = parity.golden_batch(gold, name, device="cuda")
    ag.change_morphology(g)
    names = [str(s) for s in gold["state_names"]]
    for it in range(2):
        before = agent_state(ag)
        ld = ag.update(b, it, noise=torch.tensor(gold[name + "/noise"][it], device="cuda"))
        want = float(gold[name + f"/upd{it}/critic_loss"])
        assert abs(ld["loss/critic_loss"].item() - want) < 1e-4 * want
        assert ("loss/actor_loss" in ld) == (it == 0)
        if it == 0:
            wa = float(gold[name + "/upd0/actor_loss"])
            assert abs(ld["loss/actor_loss"].item() - wa) < 1e-4 * abs(wa)
        assert abs(ld["misc/train_reward_mean"] - float(gold[name + f"/upd{it}/reward_mean"])) < 1e-6
        assert abs(ld["misc/train_reward_var"] - float(gold[name + f"/upd{it}/reward_var"])) < 1e-6
        after = agent_state(ag)
        step = {n: after[n] - before[n] for n in names}
        parity.check_summary(parity.summarize(step), gold[name + f"/upd{it}/step"], rtol=2e-3, floor=1e-3, what=f"step it={it}")
    with torch.no_grad():
        assert parity.rel_err(ag.actor(b["obs"]), gold[name + "/actions_after"]) < parity.RTOL
        assert parity.rel_err(ag.critic_target.Q1(b["obs"], b["action"]), gold[name + "/tq1_after"]) < parity.RTOL


def test_four_updates_match_oracle_humanoid_b100():
    """k=4 consecutive updates at a BASELINE size vs the oracle TD3 step (torch Adam, clip_grad_norm_,
    Polyak) run on the same GPU.  Losses/targets are checked against an fp64 oracle at 1e-4; the
    parameter trajectories against an fp32 oracle (Adam's sign-like first steps and the few-ulp
    Polyak increments make fp32-vs-fp64 trajectories differ by ~1e-2 even for the reference itself)."""
    ag, pa, pc = make_agent()
    par = M.ALL["3d_humanoid_9_full"]
    g = G.build_graph(par, device="cuda")
    ag.change_morphology(g)
    B = 100
    g64 = dict(g); g64["relation"] = g["relation"].double()
    td64 = O.TD3Oracle({k: v.cuda().double() for k, v in pa.items()}, {k: v.cuda().double() for k, v in pc.items()})
    td32 = O.TD3Oracle({k: v.cuda() for k, v in pa.items()}, {k: v.cuda() for k, v in pc.items()})
    for it in range(4):
        b = {k: v.cuda() for k, v in synth.make_batch(B, len(par), seed=20 + it).items()}
        noise = torch.randn(B, 27, generator=torch.Generator().manual_seed(it)).cuda() * 0.2
        ld = ag.update(b, it, noise=noise)
        ref = td64.update({k: v.double() for k, v in b.items()}, it, noise.double(), g64)
        td32.update(b, it, noise, g)
        assert abs(ld["loss/critic_loss"].item() - ref["loss/critic_loss"].item()) < 1e-4 * ref["loss/critic_loss"].item()
        assert parity.rel_err(ag._last_target, ref["target_Q"].reshape(-1)) < 2e-4      # after k steps the nets themselves differ slightly
        if it % 2 == 0:
            assert abs(ld["loss/actor_loss"].item() - ref["loss/actor_loss"].item()) < 5e-4 * abs(ref["loss/actor_loss"].item())

    def traj_err(mod, ref_p, init):
        num = den = 0.0
        for k, p in mod.named_parameters():
            d0 = init[k].cuda().double()
            num += ((p.double() - d0) - (ref_p[k].detach().double() - d0)).pow(2).sum().item()
            den += (ref_p[k].detach().double() - d0).pow(2).sum().item()
        return (num / den) ** 0.5

    noise_floor = max(traj_err(ag.critic, td64.critic, pc), 1e-3)     # fp32-vs-fp64 scale of this trajectory
    for mod, r32, init, what in ((ag.critic, td32.critic, pc, "critic"), (ag.actor, td32.actor, pa, "actor"),
                                 (ag.critic_target, td32.critic_t, pc, "critic_target"), (ag.actor_target, td32.actor_t, pa, "actor_target")):
        e = traj_err(mod, r32, init)
        assert e < 3e-2, (what, e, noise_floor)
    # and the fp32 oracle is itself that far from fp64: our trajectory is not worse than 3x the reference arithmetic's own noise
    ref_noise = traj_err_dict(td32.critic, td64.critic, pc)
    assert traj_err(ag.critic, td64.critic, pc) < 3 * max(ref_noise, 1e-3), (traj_err(ag.critic, td64.critic, pc), ref_noise)
    assert int(ag.critic_optimizer.step_count.item()) == 4 and int(ag.actor_optimizer.step_count.item()) == 2
    with torch.no_grad():
        b = {k: v.cuda() for k, v in synth.make_batch(B, len(par), seed=99).items()}
        assert parity.rel_err(ag.actor(b["obs"]), O.actor_forward(td64.actor, b["obs"].double(), g64)) < 1e-3
        assert parity.rel_err(ag.critic(b["obs"], b["action"])[0], O.critic_forward(td64.critic, b["obs"].double(), b["action"].double(), g64)[0]) < 1e-3


def traj_err_dict(a, b, init):
    num = den = 0.0
    for k in a:
        d0 = init[k].cuda().double()
        num += ((a[k].detach().double() - d0) - (b[k].detach().double() - d0)).pow(2).sum().item()
        den += (b[k].detach().double() - d0).pow(2).sum().item()
    return (num / den) ** 0.5


def test_select_action_matches_forward():
    ag, pa, _ = make_agent()
    par = M.ALL["3d_walker_7_full"]
    g = G.build_graph(par, device="cuda")
    ag.change_morphology(g)
    obs = synth.make_obs(1, len(par), seed=4)[0].numpy().astype(np.float64)
    a = ag.select_action(obs)
    assert isinstance(a, np.ndarray) and a.shape == (1, 3 * len(par)) and a.dtype == np.float32
    ref = O.actor_forward(pa, torch.tensor(obs, dtype=torch.float32)[None], G.build_graph(par))
    assert parity.rel_err(a, ref) < parity.RTOL


def _arena_grads(mod):
    """{name: gradient view} out of a module's flat gradient arena (what Agent.update's backward kernels wrote)."""
    names = {id(p): k for k, p in mod.named_parameters()}
    ga, live = mod.grad_arena(), mod._nb * mod._live
    return {names[id(p)]: (ga[a:a + n].view(p.shape) if a < live else None) for p, a, n in mod._slots}


@pytest.mark.parametrize("B", [100, 256])
def test_replayed_graph_gradients_equal_eager_gradients(B):
    """Race detector for the captured update: two agents with identical state take the same eight steps (humanoid-9,
    B=100, the size where a cross-stream ordering hazard once showed, and B=256, the benched size), one replaying the captured CUDA graphs
    (iterations 2-7), the other running every launch eagerly.  The forward passes are deterministic and the only
    run-to-run freedom in the backward is the order of the split-K atomics (~1e-7), so the raw gradients of both must
    agree far below the parity bar; a forked weight-gradient GEMM reading a half-written dY would not.

    The actor gradient of a step is taken through the critic as that step's own Adam update left it, and the two agents'
    critics differ there by the atomics order of their critic gradients (~1e-10).  That is enough to put a relu unit of the
    actor step's critic forward on the other side of its kink now and then, which moves the actor gradient by a share of one
    sample (2e-5 at B=256).  So the eager actor gradient it is compared with comes from a third agent, eager as well, that
    starts the step from the same state but with the replaying agent's updated critic and a critic learning rate of 0: both
    actor gradients then go through bit-identical forward passes.

    (Comparing LATER steps tensor by tensor against an fp64 oracle is not meaningful: of the ~6 M relu evaluations of a
    step a handful have |pre-activation| < 1e-6 of their row scale, and their sign - hence a gradient contribution of up
    to 1e-2 of one sample - is decided by fp32 summation order; tools/debug_relu_masks.py lists them.  Fresh-weight
    gradients are checked against the oracle in tests/test_backward_gpu.py.)"""
    ag, _, _ = make_agent()
    eg, _, _ = make_agent()
    xg, _, _ = make_agent()
    eg.use_graphs = xg.use_graphs = False
    par = M.ALL["3d_humanoid_9_full"]
    g = G.build_graph(par, device="cuda")
    ag.change_morphology(g); eg.change_morphology(g); xg.change_morphology(g)
    for it in range(8):
        # both start every step from bit-identical state (the atomics-order noise of the previous step would otherwise grow,
        # through a relu kink, into a 1e-4 difference within a few steps)
        for other in (eg, xg):
            other.load_state_dict(ag.state_dict())
            other.critic_optimizer.load_state_dict(ag.critic_optimizer.state_dict())
            other.actor_optimizer.load_state_dict(ag.actor_optimizer.state_dict())
        b = {k: v.cuda() for k, v in synth.make_batch(B, len(par), seed=50 + it).items()}
        noise = torch.randn(B, 27, generator=torch.Generator().manual_seed(100 + it)).cuda() * 0.2
        la, le = ag.update(b, it, noise=noise), eg.update(b, it, noise=noise)
        assert abs(la["loss/critic_loss"].item() - le["loss/critic_loss"].item()) <= 1e-6 * abs(le["loss/critic_loss"].item()), it
        assert parity.rel_err(ag.critic.grad_arena(), eg.critic.grad_arena()) < 1e-5, it
        if it % 2 == 0:
            xg.critic.load_state_dict(ag.critic.state_dict())
            xg.critic_optimizer.lr = 0.0
            xg.update(b, it, noise=noise)
            assert torch.equal(xg.critic.full_arena, ag.critic.full_arena), it
            assert parity.rel_err(ag.actor.grad_arena(), xg.actor.grad_arena()) < 1e-5, it
        for ma, me in ((ag.critic, eg.critic), (ag.actor, eg.actor), (ag.critic_target, eg.critic_target)):
            assert parity.rel_err(ma.full_arena, me.full_arena) < 1e-5, it     # one Adam sign flip of a ~0 gradient entry moves this by ~2e-6
    plan = next(iter(ag._plans.values()))
    assert set(plan.graphs) == {(True, False), (False, False)} and not eg._plans[next(iter(eg._plans))].graphs


def test_weights_written_from_python_reach_the_tensor_core_path():
    """ADVICE r01 (modules.py tf32 split): the tcgen05 GEMMs stream a pre-split copy (hi/lo) of the weights that the fused
    Adam / Polyak kernels keep in sync.  Every torch-side write must stale it: after a move (.cpu().cuda() re-flattens the
    arena, so the parameters stop sharing the arena's version counter), load_state_dict, an in-place p.copy_ and — with the
    documented invalidate_split() — a write through p.data.  Agent A goes through those edits between updates; agent B is
    built fresh with the same weights and optimizer state each time; their next update must agree."""
    par = M.ALL["3d_humanoid_9_full"]
    g = G.build_graph(par, device="cuda")
    B = 100
    a, _, _ = make_agent()
    a = a.cpu().cuda()                                   # forces _reflatten: per-parameter version counters from here on
    a.change_morphology(g)
    other = {k: v + 0.01 * torch.randn(v.shape, generator=torch.Generator().manual_seed(len(k))).to(v.device)
             for k, v in agent_state(a).items()}

    def edits():
        yield "load_state_dict", lambda: a.load_state_dict(other)
        def inplace():
            with torch.no_grad():
                for p in a.critic.parameters():
                    p.mul_(1.001)
        yield "in-place p.mul_", inplace
        def through_data():
            for p in a.actor.parameters():
                p.data.copy_(p.data * 0.999)
            a.actor.invalidate_split()
        yield "p.data + invalidate_split", through_data

    it = 0
    for what, edit in edits():
        b = {k: v.cuda() for k, v in synth.make_batch(B, len(par), seed=70 + it).items()}
        noise = torch.randn(B, 27, generator=torch.Generator().manual_seed(7 + it)).cuda() * 0.2
        a.update(b, it, noise=noise); a.update(b, it + 1, noise=noise)        # split fresh and trusted, graphs captured or replayed
        edit()
        fresh, _, _ = make_agent()
        fresh.change_morphology(g)
        fresh.load_state_dict(a.state_dict())
        fresh.critic_optimizer.load_state_dict(a.critic_optimizer.state_dict())
        fresh.actor_optimizer.load_state_dict(a.actor_optimizer.state_dict())
        la, lf = a.update(b, it + 2, noise=noise), fresh.update(b, it + 2, noise=noise)
        assert abs(la["loss/critic_loss"].item() - lf["loss/critic_loss"].item()) <= 1e-6 * abs(lf["loss/critic_loss"].item()), what
        assert parity.rel_err(a.critic.grad_arena(), fresh.critic.grad_arena()) < 1e-5, what
        assert parity.rel_err(a.actor.grad_arena(), fresh.actor.grad_arena()) < 1e-4, what
        it += 2
