"""Per-seed TD3 hyper-parameters of SeedBatchedAgent without a GPU: the overrides are validated (and in which order the errors
come), get_hparams / set_hparams round-trip, agent(k) and from_agents carry each seed's values into args and the optimizers,
from_agents refuses agents that differ in a value the seeds share, and the rows of the device table are rounded like the
by-value arguments they replace.  The step itself is in test_seed_hparams_gpu.py."""
import math

import numpy as np
import pytest
import torch

from oracle import ref_loader

KEYS = ("actor_lr", "critic_lr", "discount", "policy_noise", "noise_clip", "grad_clipping_value", "target_smoothing_tau", "reward_scale")


def _args():
    return ref_loader.default_args()


def _from_args(a):
    return dict(actor_lr=a.lr, critic_lr=a.lr, discount=a.discount, policy_noise=a.policy_noise, noise_clip=a.noise_clip,
                grad_clipping_value=a.grad_clipping_value, target_smoothing_tau=a.agent.target_smoothing_tau,
                reward_scale=a.agent.reward_scale)


SWEEP = [dict(lr=3e-4), dict(actor_lr=1e-4, critic_lr=2e-4, discount=0.97, policy_noise=0.1, noise_clip=0.3, grad_clipping_value=0.0,
                             target_smoothing_tau=0.01, reward_scale=2.0),
         dict(lr=5e-4, critic_lr=7e-4, target_smoothing_tau=1.0)]


def test_no_hparams_gives_every_seed_args_values():
    from sgrl_b200.seed_batch import HPARAM_KEYS, SeedBatchedAgent
    assert HPARAM_KEYS == KEYS
    args = _args()
    args.discount, args.agent.reward_scale = 0.95, 3.0
    sb = SeedBatchedAgent(args, [1, 2, 3])
    for k in range(3):
        assert sb.get_hparams(k) == pytest.approx(_from_args(args), rel=0, abs=0)


def test_hparams_override_args_per_seed():
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), [1, 2, 3], hparams=SWEEP)
    base = _from_args(_args())
    assert sb.get_hparams(0) == {**base, "actor_lr": 3e-4, "critic_lr": 3e-4}
    assert sb.get_hparams(1) == {**base, **SWEEP[1]}
    assert sb.get_hparams(2) == {**base, "actor_lr": 5e-4, "critic_lr": 7e-4, "target_smoothing_tau": 1.0}   # specific key wins over lr


@pytest.mark.parametrize("bad,match", [
    ({"policy_freq": 3}, "'policy_freq' is shared"),
    ({"max_action": 2.0}, "'max_action' is shared"),
    ({"batch_size": 64}, "'batch_size' is shared"),
    ({"attention_layers": 2}, "'attention_layers' is shared"),
    ({"learning_rate": 1e-3}, "unknown hyper-parameter 'learning_rate'"),
    ({"betas": 0.5}, "unknown hyper-parameter 'betas'"),
    ({"discount": float("nan")}, "discount must be a finite real number"),
    ({"lr": float("inf")}, "lr must be a finite real number"),
    ({"reward_scale": "1.0"}, "reward_scale must be a finite real number"),
    ({"discount": True}, "discount must be a finite real number"),
    ({"lr": -1e-4}, "lr must be >= 0"),
    ({"critic_lr": -1.0}, "critic_lr must be >= 0"),
    ({"grad_clipping_value": -0.1}, "grad_clipping_value must be >= 0"),
    ({"policy_noise": -0.2}, "policy_noise must be >= 0"),
    ({"noise_clip": -0.5}, "noise_clip must be >= 0"),
    ({"target_smoothing_tau": 1.5}, r"target_smoothing_tau must lie in \[0, 1\]"),
    ({"target_smoothing_tau": -0.1}, r"target_smoothing_tau must lie in \[0, 1\]"),
    # several faults: shared key first, then unknown key, then non-finite values, then ranges
    ({"lr": -1.0, "discount": float("nan"), "foo": 1, "policy_freq": 1}, "'policy_freq' is shared"),
    ({"lr": -1.0, "discount": float("nan"), "foo": 1}, "unknown hyper-parameter 'foo'"),
    ({"lr": -1.0, "discount": float("nan")}, "discount must be a finite"),
])
def test_validation_errors_and_their_order(bad, match):
    from sgrl_b200.seed_batch import SeedBatchedAgent
    torch.manual_seed(5)
    before = torch.rand(2)
    torch.manual_seed(5)
    with pytest.raises(ValueError, match=match):
        SeedBatchedAgent(_args(), [1, 2], hparams=[{}, bad])
    assert torch.equal(torch.rand(2), before)
    sb = SeedBatchedAgent(_args(), [1, 2])
    want = sb.get_hparams(1)
    with pytest.raises(ValueError, match=match):
        sb.set_hparams(1, **bad)
    assert sb.get_hparams(1) == want                      # nothing changed


def test_hparams_list_and_index_errors():
    from sgrl_b200.seed_batch import SeedBatchedAgent
    with pytest.raises(ValueError, match="1 to 8"):                       # the seed count is checked first
        SeedBatchedAgent(_args(), [], hparams=[{}])
    with pytest.raises(ValueError, match=r"one dict per seed \(2\), got 1"):
        SeedBatchedAgent(_args(), [1, 2], hparams=[{}])
    with pytest.raises(ValueError, match="expected a dict"):
        SeedBatchedAgent(_args(), [1, 2], hparams=[{}, 0.1])
    sb = SeedBatchedAgent(_args(), [1, 2])
    for call in (lambda: sb.get_hparams(2), lambda: sb.set_hparams(-1, lr=1e-3)):
        with pytest.raises(ValueError, match="seed index"):
            call()


def test_get_set_round_trip():
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), [1, 2, 3])
    before = [sb.get_hparams(k) for k in range(3)]
    sb.set_hparams(1, lr=2e-3, discount=0.9, grad_clipping_value=0.0)
    sb.set_hparams(2, target_smoothing_tau=0.02, reward_scale=np.float32(0.5))
    assert sb.get_hparams(0) == before[0]
    assert sb.get_hparams(1) == {**before[1], "actor_lr": 2e-3, "critic_lr": 2e-3, "discount": 0.9, "grad_clipping_value": 0.0}
    assert sb.get_hparams(2) == {**before[2], "target_smoothing_tau": 0.02, "reward_scale": 0.5}
    got = sb.get_hparams(2)
    got["discount"] = 0.0                                  # a copy
    assert sb.get_hparams(2)["discount"] == before[2]["discount"]


def test_agent_k_and_from_agents_carry_each_seeds_values():
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import SeedBatchedAgent
    args = _args()
    sb = SeedBatchedAgent(args, [1, 2, 3], hparams=SWEEP)
    for k in range(3):
        h = sb.get_hparams(k)
        a = sb.agent(k)
        assert a.actor_optimizer.lr == h["actor_lr"] and a.critic_optimizer.lr == h["critic_lr"]
        assert (a.args.discount, a.args.policy_noise, a.args.noise_clip, a.args.grad_clipping_value) == \
               (h["discount"], h["policy_noise"], h["noise_clip"], h["grad_clipping_value"])
        assert (a.target_smoothing_tau, a.reward_scale) == (h["target_smoothing_tau"], h["reward_scale"])
        assert (a.args.agent.target_smoothing_tau, a.args.agent.reward_scale) == (h["target_smoothing_tau"], h["reward_scale"])
        assert a.args.lr == (h["actor_lr"] if h["actor_lr"] == h["critic_lr"] else args.lr)
        assert a._seed_hparams()[0] == h
    assert (args.discount, args.agent.reward_scale, args.lr) == (0.99, 1.0, 1e-4)     # the caller's args are left alone
    # from_agents takes each agent's own values, including ones changed on the agent after it was built
    agents = [sb.agent(k) for k in range(3)]
    agents[0].critic_optimizer.lr = 9e-4
    agents[2].reward_scale = 4.0
    back = SeedBatchedAgent.from_agents(agents)
    for k in range(3):
        assert back.get_hparams(k) == agents[k]._seed_hparams()[0]
    assert back.get_hparams(0)["critic_lr"] == 9e-4 and back.get_hparams(2)["reward_scale"] == 4.0
    plain = SeedBatchedAgent.from_agents([Agent(_args()), Agent(_args())])
    assert plain.get_hparams(0) == plain.get_hparams(1) == _from_args(_args())


@pytest.mark.parametrize("key,value", [("policy_freq", 3), ("max_action", 2.0)])
def test_from_agents_refuses_mixed_shared_values(key, value):
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import SeedBatchedAgent
    a, b = Agent(_args()), Agent(ref_loader.default_args(**{key: value}))
    with pytest.raises(ValueError, match=f"{key} differ"):
        SeedBatchedAgent.from_agents([a, b])


def test_table_rows_round_like_the_by_value_arguments():
    """The rows the kernels read: fp32 fields rounded like ctypes.c_float, one_minus_tau = (float)(1.0 - (double)tau)."""
    import ctypes
    from sgrl_b200._lib import TD3_HPARAMS
    from sgrl_b200.agent import hparam_table
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), [1, 2, 3], hparams=SWEEP)
    rows = hparam_table(sb._seed_hparams())
    assert rows.dtype == TD3_HPARAMS and rows.dtype.itemsize == 48 and len(rows) == 3
    assert [rows.dtype.fields[f][1] for f in ("actor_lr", "critic_lr", "discount", "tau", "max_norm")] == [0, 8, 16, 32, 40]
    f32 = lambda x: ctypes.c_float(x).value
    for k in range(3):
        h = sb.get_hparams(k)
        assert rows["actor_lr"][k] == h["actor_lr"] and rows["critic_lr"][k] == h["critic_lr"]
        for field, key in (("discount", "discount"), ("reward_scale", "reward_scale"), ("policy_noise", "policy_noise"),
                           ("noise_clip", "noise_clip"), ("tau", "target_smoothing_tau"), ("max_norm", "grad_clipping_value")):
            assert float(rows[field][k]) == f32(h[key]), (k, field)
        assert float(rows["one_minus_tau"][k]) == f32(1.0 - f32(h["target_smoothing_tau"]))
    assert math.isclose(float(rows["one_minus_tau"][0]), 0.995, rel_tol=1e-7)
