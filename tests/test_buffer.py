"""Device-resident replay buffer (sgrl_b200/buffer.py, csrc/replay.cuh) vs the numpy restatement of
src/common/buffer.py (oracle/replay_oracle.py) and, when present, the unmodified reference class."""
import os
import random
import sys
import types

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle.replay_oracle import ReplayOracle
import parity

OD, AD = 41 * 3, 3 * 3


class _Box:
    def __init__(self, n):
        self.shape = (n,)


def _transitions(n, seed, od=OD, ad=AD):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        yield (rng.standard_normal(od).astype(np.float32), rng.uniform(-1, 1, ad).astype(np.float32),
               rng.standard_normal(od).astype(np.float32), float(rng.standard_normal()), float(rng.random() < 0.1))


def _fill(bufs, n, seed, **kw):
    for t in _transitions(n, seed, **kw):
        for b in bufs:
            b.add_transition(*t)


def _equal_storage(buf, orc):
    assert (buf.curr, buf.max_sample_size, buf.max_buffer_size) == (orc.curr, orc.max_sample_size, orc.max_buffer_size)
    for k in ("obs", "action", "next_obs", "reward", "done"):
        np.testing.assert_array_equal(getattr(buf, k + "_buffer"), getattr(orc, k + "_buffer"), err_msg=k)


# ---------------------------------------------------------------------------- oracle pinned to the reference
@pytest.mark.skipif(ref_loader.find_reference() is None, reason="reference not on this machine")
def test_oracle_against_reference_buffer():
    ref_loader.load_reference()
    import gym  # the stub package registered by ref_loader
    box_mod = sys.modules["gym.spaces.box"]
    box_mod.Box = _Box
    gym.spaces.box = box_mod
    gym.spaces.discrete = sys.modules["gym.spaces.discrete"]
    gym.spaces.discrete.Discrete = type("Discrete", (), {})
    from common.buffer import ReplayBuffer as RefBuffer  # type: ignore
    ref = RefBuffer(_Box(OD), _Box(AD - 3), max_buffer_size=37, modular=True)
    orc = ReplayOracle(OD, AD, 37)
    _fill((ref, orc), 90, seed=5)                      # wraps twice
    _equal_storage(ref, orc)
    for kw in ({}, {"sequential": True}, {"allow_duplicate": True}):
        random.seed(3); np.random.seed(4)
        want = ref.sample(16, to_tensor=False, **kw)
        random.seed(3); np.random.seed(4)
        got = orc.sample(16, **kw)
        for k in want:
            np.testing.assert_array_equal(got[k], want[k], err_msg=f"{k} {kw}")
    want = ref.get_batch([0, 5, 36, 5], to_tensor=False)
    got = orc.get_batch([0, 5, 36, 5])
    for k in want:
        np.testing.assert_array_equal(got[k], want[k])


def test_oracle_against_pins():
    """The oracle's storage, seeded samples and get_batch vs tests/golden/pins.npz.  Those were recorded from the oracle
    itself (tests/golden/make_pins.py), not from the reference class: where the reference is not available they still
    catch any change to the behaviour the device buffer is checked against."""
    from golden.make_pins import AD as PAD, CAP, OD as POD, buffer_draws
    pins = np.load(os.path.join(os.path.dirname(parity.GOLDEN), "pins.npz"))
    got = buffer_draws(ReplayOracle(POD, PAD, CAP))
    assert sorted(got) == sorted(k for k in pins.files if k.startswith("buffer/"))
    for k, v in got.items():
        np.testing.assert_array_equal(v, pins[k], err_msg=k)


# ---------------------------------------------------------------------------- host logic (no GPU needed)
def test_host_logic_matches_oracle_on_cpu_storage():
    from sgrl_b200.buffer import ReplayBuffer
    from sgrl_b200._lib import SgrlError
    ReplayBuffer.STAGE_ROWS, keep = 8, ReplayBuffer.STAGE_ROWS          # several flushes, one of them across the wrap
    try:
        buf = ReplayBuffer(_Box(OD), _Box(AD - 3), max_buffer_size=37, modular=True, device="cpu")
    finally:
        ReplayBuffer.STAGE_ROWS = keep
    orc = ReplayOracle(OD, AD, 37)
    assert (buf.obs_dim, buf.action_dim, buf.row_floats) == (OD, AD, 2 * OD + AD + 2)
    for n in (5, 20, 30, 41):
        _fill((buf, orc), n, seed=n)
        _equal_storage(buf, orc)
    for kw in ({}, {"sequential": True}, {"allow_duplicate": True}):
        random.seed(9); np.random.seed(10)
        a = list(buf.draw_indices(16, **kw))
        random.seed(9); np.random.seed(10)
        b = list(orc.draw_indices(16, **kw))
        assert a == b
    small = ReplayBuffer(OD, AD, max_buffer_size=50, device="cpu")
    _fill((small,), 7, seed=1)
    with pytest.warns(UserWarning, match="larger than buffer"):
        assert len(small.draw_indices(16)) == 7                        # buffer.py:88-91
    # snapshot interface: arrays can be assigned back (common/trainer.py:307-320)
    other = ReplayBuffer(OD, AD, max_buffer_size=37, device="cpu")
    for k in ("obs", "action", "next_obs", "reward", "done"):
        setattr(other, k + "_buffer", getattr(orc, k + "_buffer"))
    other.curr, other.max_sample_size = orc.curr, orc.max_sample_size
    _equal_storage(other, orc)
    buf.resize(60); assert buf.max_buffer_size == 60 and buf.rows.shape[0] == 60 and buf.curr == 37
    buf.resize(20); assert buf.max_buffer_size == 20 and buf.curr == 0 and buf.max_sample_size == 20
    buf.clear(); assert (buf.curr, buf.max_sample_size) == (0, 0)
    with pytest.warns(UserWarning, match="larger than buffer"):
        empty = buf.sample(4)                                           # nothing stored: an empty batch, no kernel call
    assert empty["obs"].shape == (0, OD) and empty["reward"].shape == (0, 1)
    if not torch.cuda.is_available():
        with pytest.raises(SgrlError, match="CUDA"):                    # no CPU fallback for the data path
            other.sample(4)
    with pytest.raises(NotImplementedError):
        ReplayBuffer(_Box(OD), types.SimpleNamespace(n=4))             # discrete action spaces are not part of the SET path


# ---------------------------------------------------------------------------- GPU parity (bit-exact: pure data movement)
@pytest.mark.gpu
@pytest.mark.parametrize("n_limbs,cap,n_add", [(3, 37, 90), (9, 1000, 700), (2, 64, 64)])
def test_sample_parity_gpu(n_limbs, cap, n_add):
    from sgrl_b200.buffer import ReplayBuffer
    od, ad = 41 * n_limbs, 3 * n_limbs
    buf = ReplayBuffer(od, ad, max_buffer_size=cap)
    orc = ReplayOracle(od, ad, cap)
    assert buf.rows.is_cuda
    _fill((buf, orc), n_add, seed=n_limbs, od=od, ad=ad)
    _equal_storage(buf, orc)
    for kw in ({}, {"sequential": True}, {"allow_duplicate": True}):
        for B in (1, 16, min(256, orc.max_sample_size)):
            random.seed(B); np.random.seed(B + 1)
            got = buf.sample(B, **kw)
            random.seed(B); np.random.seed(B + 1)
            want = orc.sample(B, **kw)
            for k in want:
                assert got[k].is_cuda and got[k].dtype == torch.float32 and tuple(got[k].shape) == want[k].shape, (k, got[k].shape)
                np.testing.assert_array_equal(got[k].cpu().numpy(), want[k], err_msg=f"{k} {kw} B={B}")
    idx = [0, cap - 1, 3, 3, -1]
    got, want = buf.get_batch(idx), orc.get_batch(idx)
    assert tuple(got["reward"].shape) == (5, 1, 1)                      # buffer.py:143-144 (reshape + unsqueeze)
    for k in want:
        np.testing.assert_array_equal(got[k].cpu().numpy().reshape(want[k].shape), want[k])
    host = buf.sample(8, to_tensor=False)
    assert isinstance(host["obs"], np.ndarray) and host["reward"].shape == (8, 1)
    with pytest.raises(IndexError):
        buf.get_batch([cap])
    # transitions that are already on the device
    more = list(_transitions(11, seed=77, od=od, ad=ad))
    for t in more:
        orc.add_transition(*t)
    cols = [torch.tensor(np.stack([np.atleast_1d(np.asarray(t[i], dtype=np.float32)) for t in more])).cuda() for i in range(5)]
    buf.add_batch(*cols)
    _equal_storage(buf, orc)


@pytest.mark.gpu
def test_update_from_buffer_equals_update_of_sampled_batch():
    from oracle import set_oracle as O
    from sgrl_b200 import graph as G, morphologies as M, synth
    from sgrl_b200.agent import Agent
    from sgrl_b200.buffer import ReplayBuffer
    from sgrl_b200.config import default_args
    par = M.ALL["3d_walker_7_full"]
    n, B = len(par), 32
    g = G.build_graph(par, device="cuda")
    data = synth.make_batch(300, n, seed=5)
    agents = []
    for _ in range(2):
        torch.manual_seed(0)
        ag = Agent(default_args())
        ag.change_morphology(g)
        agents.append(ag)
    buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=256)
    for i in range(300):                                                # wraps once
        buf.add_transition(data["obs"][i].numpy(), data["action"][i].numpy(), data["next_obs"][i].numpy(),
                           float(data["reward"][i]), float(data["done"][i]))
    noise = torch.randn(B, 3 * n, device="cuda") * 0.2
    for it in range(4):
        random.seed(100 + it)
        l0 = agents[0].update_from_buffer(buf, B, it, noise=noise)
        random.seed(100 + it)
        l1 = agents[1].update(buf.sample(B), it, noise=noise)
        assert abs(l0["loss/critic_loss"].item() - l1["loss/critic_loss"].item()) <= 1e-5 * abs(l1["loss/critic_loss"].item())
        assert abs(l0["misc/train_reward_mean"] - l1["misc/train_reward_mean"]) < 1e-6
    for m0, m1 in ((agents[0].critic, agents[1].critic), (agents[0].actor, agents[1].actor), (agents[0].actor_target, agents[1].actor_target)):
        assert parity.rel_err(m0.full_arena, m1.full_arena) < 1e-5     # same inputs; only split-K atomics reorder sums (one Adam sign flip of a ~0 gradient entry moves this by ~2e-6)
    with pytest.raises(ValueError, match="morphology"):
        agents[0].change_morphology(G.build_graph(M.ALL["3d_hopper_3_shin"], device="cuda"))
        agents[0].update_from_buffer(buf, B, 0)
