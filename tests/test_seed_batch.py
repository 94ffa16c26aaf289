"""Seed-batched TD3 without a GPU (sgrl_b200.seed_batch): each seed's initial weights are those of
``torch.manual_seed(seed); Agent(args)`` bit for bit, the modules build on the CPU, arguments are validated, and agent(k) /
from_agents round-trip the reference's 818 state_dict keys and the Adam state.  The step itself is in test_seed_batch_gpu.py."""
import pytest
import torch

from oracle import ref_loader

MODS = ("actor", "critic", "actor_target", "critic_target")


def _args():
    return ref_loader.default_args()


def test_initial_weights_are_the_seeds_agents():
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import SeedBatchedAgent
    seeds = [4, 17, 4]
    torch.manual_seed(99)
    before = torch.rand(3)
    torch.manual_seed(99)
    sb = SeedBatchedAgent(_args(), seeds)
    assert torch.equal(torch.rand(3), before)                   # the caller's random stream is left alone
    assert sb.n_seeds == 3 and sb.actor._nb == 3 and sb.critic._nb == 6
    for k, s in enumerate(seeds):
        torch.manual_seed(s)
        want = Agent(_args())
        got = sb.agent(k)
        for m in MODS:
            assert torch.equal(getattr(got, m).full_arena, getattr(want, m).full_arena), (k, m)
        sd_got, sd_want = got.state_dict(), want.state_dict()
        assert len(sd_want) == 818 and list(sd_got) == list(sd_want)
        assert all(torch.equal(sd_got[x], sd_want[x]) for x in sd_want)
    # critic nets in seed-batched order: [critic1 of every seed | critic2 of every seed]
    L = sb.critic._live
    c = sb.agent(1).critic.live_arena
    assert torch.equal(sb.critic.live_arena[1 * L:2 * L], c[:L]) and torch.equal(sb.critic.live_arena[4 * L:5 * L], c[L:])


def test_argument_validation():
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import SeedBatchedAgent
    for seeds in ([], list(range(9))):
        with pytest.raises(ValueError, match="1 to 8"):
            SeedBatchedAgent(_args(), seeds)
    sb = SeedBatchedAgent(_args(), [1, 2])
    with pytest.raises(ValueError, match="one per seed"):
        sb.update([{}], 0)
    with pytest.raises(ValueError, match="one per seed"):
        sb.update([{}, {}, {}], 0)
    with pytest.raises(ValueError, match="one per seed"):
        sb.select_actions([[]], [])
    with pytest.raises(ValueError, match="seed index"):
        sb.agent(2)
    with pytest.raises(NotImplementedError):
        sb.update_packed([], 0)
    with pytest.raises(ValueError, match="1 to 8"):
        SeedBatchedAgent.from_agents([])
    a, b = Agent(_args()), Agent(_args())
    b.critic_optimizer.step_count += 1
    with pytest.raises(ValueError, match="step counts differ"):
        SeedBatchedAgent.from_agents([a, b])


def test_from_agents_and_agent_round_trip():
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import SeedBatchedAgent
    agents = []
    for s in (3, 8, 5):
        torch.manual_seed(s)
        a = Agent(_args())
        g = torch.Generator().manual_seed(s)
        for opt in (a.actor_optimizer, a.critic_optimizer):      # distinct optimizer state per seed
            opt.exp_avg.copy_(torch.randn(opt.exp_avg.shape, generator=g))
            opt.exp_avg_sq.copy_(torch.rand(opt.exp_avg_sq.shape, generator=g))
            opt.step_count.fill_(7)
        a.tot_update_count = 13
        agents.append(a)
    sb = SeedBatchedAgent.from_agents(agents)
    assert sb.tot_update_count == 13
    for k, want in enumerate(agents):
        got = sb.agent(k)
        sd_got, sd_want = got.state_dict(), want.state_dict()
        assert list(sd_got) == list(sd_want) and len(sd_want) == 818
        assert all(torch.equal(sd_got[x], sd_want[x]) for x in sd_want)
        for name in ("actor_optimizer", "critic_optimizer"):
            x, y = getattr(got, name).state_dict(), getattr(want, name).state_dict()
            for key in ("step", "exp_avg", "exp_avg_sq"):
                assert torch.equal(x[key], y[key]), (k, name, key)
            assert (x["lr"], x["betas"], x["eps"]) == (y["lr"], y["betas"], y["eps"])
        assert got.tot_update_count == 13
