"""Packed multi-morphology TD3 update straight from per-morphology device replay buffers (sgrl_b200.buffer.gather_packed_into,
Agent.update_packed_from_buffers, csrc/replay.cuh): the one-launch gather over several buffers is bit-exact against the
per-buffer get_batch laid out in packed token order, and the update equals update_packed of the batches buf.sample draws with
the same seed — bit for bit in deterministic mode — on the same plan and captured graphs, with the gather as the only launch
outside the graph.  The two-rank run needs 2 GPUs and is skipped otherwise."""
import os
import random
import sys
import warnings

import numpy as np
import pytest
import torch

import parity
from sgrl_b200 import graph as G, morphologies as M, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

# one morphology per limb count the gather test covers (odd row widths: 2*41n + 3n + 2)
MORPHS = ["3d_walker_2_right_leg_left_knee", "3d_hopper_5_full", "3d_humanoid_9_full", "3d_cheetah_14_full"]


def _add_rows(buf, n, seed, host=False):
    """n synthetic transitions: host-side add_transition (left staged until the next flush) or one device add_batch."""
    b = synth.make_batch(n, buf.obs_dim // 41, seed=seed)
    if host:
        for i in range(n):
            buf.add_transition(b["obs"][i].numpy(), b["action"][i].numpy(), b["next_obs"][i].numpy(), float(b["reward"][i]),
                               float(b["done"][i]))
    else:
        buf.add_batch(*(b[k].cuda() for k in ("obs", "action", "next_obs", "reward", "done")))


def _buffers():
    """2-limb buffer wrapped, 5-limb buffer holding fewer rows than a batch, 9-limb buffer with unflushed add_transition rows
    on top of device rows, 14-limb buffer part full."""
    from sgrl_b200.buffer import ReplayBuffer
    n = [len(M.ALL[m]) for m in MORPHS]
    bufs = [ReplayBuffer(41 * k, 3 * k, max_buffer_size=cap) for k, cap in zip(n, (64, 1000, 500, 300))]
    for i in range(4):                                                # 160 rows into 64: wrapped twice
        _add_rows(bufs[0], 40, seed=1 + i)
    _add_rows(bufs[1], 20, seed=3)
    _add_rows(bufs[2], 200, seed=4)
    _add_rows(bufs[2], 37, seed=5, host=True)
    _add_rows(bufs[3], 250, seed=6)
    return bufs


def _expected(bufs, indices):
    """Per-buffer get_batch outputs concatenated: the packed token order."""
    outs = [b.get_batch(ix) for b, ix in zip(bufs, indices)]
    return {k: torch.cat([o[k].reshape(-1) for o in outs]) for k in ("obs", "action", "next_obs", "reward", "done")}


def _empty_like_packed(bufs, counts):
    f = lambda n: torch.full((n,), float("nan"), device="cuda")
    G_ = sum(counts)
    return (f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(c * b.action_dim for c, b in zip(counts, bufs))),
            f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(G_), f(G_))


def test_packed_gather_is_bit_exact():
    from sgrl_b200._lib import lib
    from sgrl_b200.buffer import gather_packed_into
    bufs = _buffers()
    assert bufs[2]._staged > 0                                       # rows the gather must flush first
    B = 32
    random.seed(7)
    with pytest.warns(UserWarning, match="larger than buffer"):
        indices = [list(b.draw_indices(B)) for b in bufs]
    assert [len(ix) for ix in indices] == [B, 20, B, B]              # the 5-limb buffer clamps its batch (buffer.py:88-91)
    for b, ix in zip(bufs, indices):
        ix += [-1, -b.max_buffer_size, b.max_buffer_size - 1]        # numpy negative indexing, last row
    counts = [len(ix) for ix in indices]
    out = _empty_like_packed(bufs, counts)
    l0 = lib.sgrl_launch_count()
    assert gather_packed_into(bufs, indices, *out) == sum(counts)
    assert lib.sgrl_launch_count() - l0 == 1
    want = _expected(bufs, indices)
    for k, got in zip(("obs", "action", "next_obs", "reward", "done"), out):
        assert torch.equal(got, want[k]), k
    # indices already on the device (the caller's own upload), given as numpy arrays
    out2 = _empty_like_packed(bufs, counts)
    flat = torch.tensor([i for ix in indices for i in ix], dtype=torch.int64, device="cuda")
    gather_packed_into(bufs, [np.asarray(ix) for ix in indices], *out2, idx_dev=flat)
    for a, b in zip(out, out2):
        assert torch.equal(a, b)
    # one part is the single-buffer gather
    one = _empty_like_packed(bufs[3:], counts[3:])
    gather_packed_into(bufs[3:], indices[3:], *one)
    for k, got in zip(("obs", "action", "next_obs", "reward", "done"), one):
        assert torch.equal(got, _expected(bufs[3:], indices[3:])[k]), k
    # out-of-range rows: the same IndexError as get_batch, raised before anything is launched
    for bad in (bufs[1].max_buffer_size, -bufs[1].max_buffer_size - 1):
        with pytest.raises(IndexError, match=f"buffer of {bufs[1].max_buffer_size} rows"):
            bufs[1].get_batch([bad])
        l0 = lib.sgrl_launch_count()
        with pytest.raises(IndexError, match=f"buffer of {bufs[1].max_buffer_size} rows"):
            gather_packed_into(bufs, [indices[0], [0, bad], indices[2], indices[3]], *_empty_like_packed(bufs, [counts[0], 2] + counts[2:]))
        assert lib.sgrl_launch_count() == l0


def _agent_parts(bufs):
    return [(G.build_graph(M.ALL[m], device="cuda"), b) for m, b in zip(MORPHS, bufs)]


def _run_pair(graphs, B, seeds):
    """Two identically built agents: one steps update_packed_from_buffers, the other update_packed on buf.sample batches,
    each after random.seed(s).  Returns per step both loss dicts, and both agents."""
    from test_agent_gpu import make_agent
    bufs = _buffers()
    parts = _agent_parts(bufs)
    agents = [make_agent()[0] for _ in range(2)]
    for ag in agents:
        ag.use_graphs = graphs
    losses = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)                 # the 5-limb buffer holds fewer rows than B
        for it, s in enumerate(seeds):
            random.seed(s)
            l0 = agents[0].update_packed_from_buffers(parts, B, it)
            st0 = random.getstate()
            random.seed(s)
            l1 = agents[1].update_packed([(g, buf.sample(B)) for g, buf in parts], it)
            assert random.getstate() == st0
            losses.append((l0, l1))
    torch.cuda.synchronize()
    return losses, agents


NETS = ("actor", "actor_target", "critic", "critic_target")


@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
def test_update_equals_update_packed_of_sampled_batches(graphs):
    from sgrl_b200._lib import lib
    prev = lib.sgrl_deterministic(1)
    try:
        losses, agents = _run_pair(graphs, 32, [11, 12, 13, 14])          # it = 0..3: both step kinds, replayed when graphs
    finally:
        lib.sgrl_deterministic(prev)
    for l0, l1 in losses:
        assert l0.keys() == l1.keys()
        for k in l0:
            a, b = l0[k], l1[k]
            assert (torch.equal(a, b) if torch.is_tensor(a) else a == b), (k, a, b)
    for name in NETS:
        assert torch.equal(getattr(agents[0], name).full_arena, getattr(agents[1], name).full_arena), name
    # the default mode sums with fp32 atomics: same inputs, the same bar as update_from_buffer vs update (test_buffer.py).  The
    # actor loss (-mean Q, a sum that nearly cancels) goes through the critic just updated with those atomics; it is compared
    # bit for bit above
    losses, agents = _run_pair(graphs, 32, [21, 22, 23, 24])
    for l0, l1 in losses:
        assert l0.keys() == l1.keys()
        for k in ("loss/critic_loss", "misc/train_reward_mean", "misc/train_reward_var"):
            a, b = float(l0[k]), float(l1[k])
            assert abs(a - b) <= 1e-5 * abs(b), (k, a, b)
    for name in NETS:
        assert parity.rel_err(getattr(agents[0], name).full_arena, getattr(agents[1], name).full_arena) < 1e-5, name


def test_one_plan_and_one_launch_per_replayed_step():
    from sgrl_b200._lib import lib
    from test_agent_gpu import make_agent
    ag = make_agent()[0]
    bufs = _buffers()
    parts = _agent_parts(bufs)
    B = 32
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for it in range(4):                                              # eager run + capture of both step kinds
            ag.update_packed_from_buffers(parts, B, it)
        plans, tables = len(ag._plans), len(ag._packed_tables)
        plan = next(reversed(ag._plans.values()))
        assert plans == 1 and tables == 1 and len(plan.graphs) == 2
        graphs = dict(plan.graphs)
        for it in range(4, 8):
            ag.update_packed([(g, buf.sample(B)) for g, buf in parts], it)
            assert (len(ag._plans), len(ag._packed_tables)) == (plans, tables)
        for it in range(8, 12):
            l0 = lib.sgrl_launch_count()
            ag.update_packed_from_buffers(parts, B, it)
            assert lib.sgrl_launch_count() - l0 == 1, it                # the gather; the step itself is the replayed graph
            assert (len(ag._plans), len(ag._packed_tables)) == (plans, tables)
        assert plan.graphs == graphs and next(reversed(ag._plans.values())) is plan
        # a resized buffer needs no new plan: the gather sits outside the graph
        bufs[3].resize(400)
        ag.update_packed_from_buffers(parts, B, 12)
        assert (len(ag._plans), len(ag._packed_tables)) == (plans, tables) and plan.graphs == graphs
    # lazy statistics stay on the device and equal the eager ones
    ag.lazy_stats = True
    random.seed(5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        lazy = ag.update_packed_from_buffers(parts, B, 13)
        assert torch.is_tensor(lazy["misc/train_reward_mean"]) and lazy["misc/train_reward_mean"].is_cuda
        ag.lazy_stats = False
        random.seed(5)
        idx = [buf.draw_indices(B) for buf in bufs]
    r = torch.cat([buf.get_batch(ix)["reward"].reshape(-1) for buf, ix in zip(bufs, idx)]).double()
    assert abs(lazy["misc/train_reward_mean"].item() - r.mean().item()) < 1e-6
    assert abs(lazy["misc/train_reward_var"].item() - r.var().item()) < 1e-5


def test_errors():
    from sgrl_b200.buffer import ReplayBuffer
    from test_agent_gpu import make_agent
    ag = make_agent()[0]
    bufs = _buffers()
    parts = _agent_parts(bufs)
    state = random.getstate()
    with pytest.raises(ValueError, match="morphology"):                 # rows of another limb count
        ag.update_packed_from_buffers([(parts[0][0], bufs[1])] + parts[1:], 8, 0)
    empty = ReplayBuffer(bufs[1].obs_dim, bufs[1].action_dim, max_buffer_size=16)
    with pytest.raises(ValueError, match="empty"):
        ag.update_packed_from_buffers(parts[:1] + [(parts[1][0], empty)], 8, 0)
    on_cpu = ReplayBuffer(bufs[1].obs_dim, bufs[1].action_dim, max_buffer_size=16, device="cpu")
    _add_rows(on_cpu, 4, seed=8, host=True)
    with pytest.raises(ValueError, match="cpu"):
        ag.update_packed_from_buffers(parts[:1] + [(parts[1][0], on_cpu)], 8, 0)
    with pytest.raises(ValueError, match="1 to 64"):
        ag.update_packed_from_buffers([parts[0]] * 65, 8, 0)
    assert random.getstate() == state                                  # nothing was drawn
    assert len(ag._plans) == 0


# ---------------------------------------------------------------------------- data parallel on 2 GPUs
def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from sgrl_b200.buffer import ReplayBuffer
        from test_agent_gpu import make_agent
        names = sorted(M.SETS["3d_humanoids"])
        mine = names[rank::world]                                      # half of Humanoid++ per rank
        parts = []
        for i, name in enumerate(mine):
            n = len(M.ALL[name])
            buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=4096, device=dev)
            b = synth.make_batch(1000, n, seed=100 * rank + i)
            buf.add_batch(*(b[k].to(dev) for k in ("obs", "action", "next_obs", "reward", "done")))
            parts.append((G.build_graph(M.ALL[name], device=dev), buf))
        ag, _, _ = make_agent()
        init = ag.critic.live_arena.clone()
        random.seed(1000 + rank)
        for it in range(6):                    # it = 0, 1 eager; 2, 3 captured; 2..5 replayed graphs
            ag.update_packed_from_buffers(parts, 64, it, morph_count=len(names) / world)
        torch.cuda.synchronize()
        sums = []
        for m in (ag.actor, ag.critic, ag.actor_target, ag.critic_target):
            bits = m.full_arena.view(torch.int32).to(torch.int64)
            sums += [bits.sum(), (bits * (torch.arange(bits.numel(), device=dev) % 8191 + 1)).sum()]
        mine_sum = torch.stack(sums)
        allv = [torch.zeros_like(mine_sum) for _ in range(world)]
        dist.all_gather(allv, mine_sum)
        same = all(bool((v == allv[0]).all()) for v in allv)
        moved = parity.rel_err(ag.critic.live_arena, init)
        replays = sum(len(p.graphs) for p in ag._plans.values())
        if rank == 0:
            out.put((same, moved, replays))
        torch.cuda.synchronize()
        dist.barrier()
    finally:
        os._exit(0)         # captured graphs hold NCCL work: leave without tearing the process group down (see bench.py)


@pytest.mark.timeout(900)
def test_two_rank_packed_buffer_updates_keep_replicas_identical():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29500 + (os.getpid() + 1000) % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    same, moved, replays = out.get(timeout=800)
    for p in procs:
        p.join(60)
    assert replays == 2                                              # both step kinds ran as captured graphs
    assert same, "replicas diverged"
    assert moved > 1e-6
