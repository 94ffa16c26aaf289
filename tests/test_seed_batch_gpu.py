"""Seed-batched TD3 (sgrl_b200.seed_batch.SeedBatchedAgent) against standalone Agents on the GPU, on both GEMM paths: every
seed's losses, reward statistics, raw gradients and parameters follow its own Agent given the same weights, batches and noise;
K = 1 in deterministic mode is the Agent's step bit for bit with the same launches; seeds do not leak into each other (a wrong
net-to-input mapping or clip grouping would show); the buffer path equals the batch path; the acting path equals each seed's
Agent.select_actions; and the launches of one step do not grow with K."""
import random
import warnings

import numpy as np
import pytest
import torch

from oracle import ref_loader
from sgrl_b200 import _lib, graph as G, morphologies as M, synth
from sgrl_b200._lib import lib

pytestmark = pytest.mark.gpu

TOL = 1e-5
HUMANOID = M.ALL["3d_humanoid_9_full"]
CHAIN15 = [-1] + list(range(14))
MODS = ("actor", "critic", "actor_target", "critic_target")


def _args():
    return ref_loader.default_args()


def _agents(seeds, use_tc):
    """A SeedBatchedAgent and, per seed, the Agent it must follow (same initial weights by construction)."""
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), seeds)
    singles = []
    for s in seeds:
        torch.manual_seed(s)
        singles.append(Agent(_args()))
    for ag in [sb] + singles:
        for m in MODS:
            getattr(ag, m).use_tc = use_tc
    return sb, singles


def _batch(B, n, seed):
    return {k: v.cuda() for k, v in synth.make_batch(B, n, seed=seed).items()}


def _noise(B, n, seed):
    return (torch.randn(B, 3 * n, generator=torch.Generator().manual_seed(seed)) * 0.2).cuda()


def _seed_slice(t, K, k, per, L):
    """Seed k's nets out of a seed-batched module's live-arena-shaped tensor (net j of seed k is net j*K + k)."""
    return torch.cat([t[(j * K + k) * L:(j * K + k + 1) * L] for j in range(per)])


def _per_tensor(kind, nets, got, want):
    """[(tensor, relative error)] over the live tensors of `nets` nets; floor: 1e-4 of the whole arena's norm."""
    table = [(n, s, o) for n, s, o, live in _lib.param_table(kind, 3) if live]
    L = _lib.arena_floats(kind, 3)[0]
    floor = 1e-4 * want.double().norm().item()
    out = []
    for z in range(nets):
        for name, shape, off in table:
            n = int(np.prod(shape))
            a, b = got[z * L + off:z * L + off + n].double(), want[z * L + off:z * L + off + n].double()
            out.append((f"net{z}.{name}", ((a - b).norm() / max(b.norm().item(), floor)).item()))
    return out


def _compare_seed(sb, k, ag, what):
    """Seed k's critic gradient tensors within TOL of its Agent's; every parameter tensor and the actor gradients, which come
    after an Adam step (it turns last-bit differences of near-zero gradient elements into lr-sized ones), within 1e-4."""
    K = sb.n_seeds
    bad = []
    for m in MODS:
        mod, one = getattr(sb, m), getattr(ag, m)
        per = one._nb
        got = _seed_slice(mod.live_arena, K, k, per, mod._live)
        bad += [(f"{m}.{n}", e) for n, e in _per_tensor(mod._kind, per, got, one.live_arena) if e > 1e-4]
    for m, tol in (("actor", 1e-4), ("critic", TOL)):
        mod, one = getattr(sb, m), getattr(ag, m)
        got = _seed_slice(mod.grad_arena(), K, k, one._nb, mod._live)
        bad += [(f"grad {m}.{n}", e) for n, e in _per_tensor(mod._kind, one._nb, got, one.grad_arena()) if e > tol]
    assert not bad, f"{what}, seed {k}: {len(bad)} tensors out of tolerance: {sorted(bad, key=lambda x: -x[1])[:8]}"


def _compare_seed_arenas(sb, k, ag, what):
    """Seed k's whole parameter arena of every module within TOL of its Agent's (relative, over the seed's nets)."""
    K = sb.n_seeds
    for m in MODS:
        mod, one = getattr(sb, m), getattr(ag, m)
        got = _seed_slice(mod.live_arena, K, k, one._nb, mod._live)
        err = ((got.double() - one.live_arena.double()).norm() / one.live_arena.double().norm()).item()
        assert err <= TOL, f"{what}, seed {k}, {m}: {err:.2e}"


CASES = [("humanoid9", HUMANOID, 100), ("walker2", M.ALL["3d_walker_2_right_leg_left_knee"], 64), ("chain15", CHAIN15, 48)]


@pytest.mark.parametrize("use_tc", [1, 0])
@pytest.mark.parametrize("graphs", [True, False])
@pytest.mark.parametrize("name,parents,B", CASES)
def test_seeds_follow_their_own_agents(name, parents, B, graphs, use_tc):
    """K = 3, four updates (two of them with the delayed actor step).  After the first update (critic and actor step) each
    seed's raw critic gradients are within 1e-5 of its own Agent's, per tensor (see _compare_seed).  The seed-batched step sums in another
    order than the single agent (split-K factors, tile variants and the clip norm's partial sums follow the net count), so
    from the second update on a relu unit sitting on its kink may land on the other side of zero in one of the two runs and
    move single gradient tensors far beyond 1e-5; what is checked there is what such a flip cannot move: every loss and
    reward statistic within 1e-4 and each module's whole parameter arena within 1e-5."""
    K, n = 3, len(parents)
    sb, singles = _agents([21, 22, 23], use_tc)
    g = G.build_graph(parents, device="cuda")
    for ag in [sb] + singles:
        ag.use_graphs = graphs
        ag.change_morphology(g)
    what = f"{name} B={B} graphs={graphs} use_tc={use_tc}"
    for it in range(4):
        batches = [_batch(B, n, 100 * k + it) for k in range(K)]
        noises = [_noise(B, n, 1000 * k + it) for k in range(K)]
        got = sb.update(batches, it, noises)
        assert len(got) == K
        for k in range(K):
            want = singles[k].update(batches[k], it, noise=noises[k])
            assert set(got[k]) == set(want)
            for key in want:
                a, b = float(got[k][key]), float(want[key])
                tol = TOL if it == 0 else 1e-4
                assert abs(a - b) <= tol * max(abs(b), 1e-6), f"{name} it {it} seed {k} {key}: {a} vs {b}"
        if it == 0:
            torch.cuda.synchronize()
            for k in range(K):
                _compare_seed(sb, k, singles[k], what + " after the first update")
    torch.cuda.synchronize()
    for k in range(K):
        _compare_seed_arenas(sb, k, singles[k], what + " after four updates")


def _run(sb, batches_per_it, noises_per_it):
    losses = []
    for it, (batches, noises) in enumerate(zip(batches_per_it, noises_per_it)):
        losses.append(sb.update(batches, it, noises))
    torch.cuda.synchronize()
    return losses, [getattr(sb, m).full_arena.clone() for m in MODS], [sb.critic.grad_arena().clone(), sb.actor.grad_arena().clone()]


@pytest.mark.parametrize("use_tc", [1, 0])
def test_one_seed_is_the_agent_bit_for_bit(use_tc):
    """K = 1 in deterministic mode: the same parameters, gradients and losses as Agent.update, and the same launches (eager
    count per step and kernels inside the captured graphs)."""
    prev = lib.sgrl_deterministic(1)
    try:
        sb, (ag,) = _agents([5], use_tc)
        g = G.build_graph(HUMANOID, device="cuda")
        sb.change_morphology(g); ag.change_morphology(g)
        B, n = 100, len(HUMANOID)
        counts = {"sb": [], "ag": []}
        for it in range(6):
            b, nz = _batch(B, n, 300 + it), _noise(B, n, 400 + it)
            l0 = lib.sgrl_launch_count()
            got = sb.update([b], it, [nz])[0]
            counts["sb"].append(lib.sgrl_launch_count() - l0)
            l0 = lib.sgrl_launch_count()
            want = ag.update(b, it, noise=nz)
            counts["ag"].append(lib.sgrl_launch_count() - l0)
            for key in want:
                assert float(got[key]) == float(want[key]), (it, key)
        torch.cuda.synchronize()
        assert counts["sb"] == counts["ag"]
        psb, pag = next(iter(sb._plans.values())), next(iter(ag._plans.values()))
        assert psb.graph_launches == pag.graph_launches and psb.graph_launches
        for m in MODS:
            assert torch.equal(getattr(sb, m).full_arena, getattr(ag, m).full_arena), m
        for m in ("actor", "critic"):
            assert torch.equal(getattr(sb, m).grad_arena(), getattr(ag, m).grad_arena()), m
            assert torch.equal(getattr(sb, m + "_optimizer").exp_avg_sq, getattr(ag, m + "_optimizer").exp_avg_sq), m
    finally:
        lib.sgrl_deterministic(prev)


def test_seeds_do_not_leak_into_each_other():
    """K = 3 in deterministic mode: two runs are bit-identical, and a different batch for seed 1 leaves seeds 0 and 2
    bit-identical (the net-to-input mapping z % K and the clip groups z % K keep seeds apart)."""
    prev = lib.sgrl_deterministic(1)
    try:
        B, n, K = 100, len(HUMANOID), 3
        g = G.build_graph(HUMANOID, device="cuda")
        data = [[_batch(B, n, 10 * it + k) for k in range(K)] for it in range(4)]
        noise = [[_noise(B, n, 50 * it + k) for k in range(K)] for it in range(4)]
        runs = []
        for variant in range(3):
            from sgrl_b200.seed_batch import SeedBatchedAgent
            sb = SeedBatchedAgent(_args(), [1, 2, 3])
            sb.change_morphology(g)
            d = [list(x) for x in data]
            if variant == 2:
                for it in range(4):
                    d[it][1] = _batch(B, n, 777 + it)
            runs.append((sb, _run(sb, d, noise)))
        (sa, (la, pa, ga)), (_, (lb, pb, gb)), (sc, (lc, pc, gc)) = runs
        assert all(torch.equal(x, y) for x, y in zip(pa + ga, pb + gb))
        assert [[float(v) for d in l for v in d.values()] for l in la] == [[float(v) for d in l for v in d.values()] for l in lb]
        for k in (0, 2):
            for m in MODS:
                mod = getattr(sa, m)
                per = mod._nb // K
                x = _seed_slice(getattr(sa, m).live_arena, K, k, per, mod._live)
                y = _seed_slice(getattr(sc, m).live_arena, K, k, per, mod._live)
                assert torch.equal(x, y), (m, k)
            for it in range(4):
                assert float(la[it][k]["loss/critic_loss"]) == float(lc[it][k]["loss/critic_loss"])
        assert not torch.equal(_seed_slice(sa.critic.live_arena, K, 1, 2, sa.critic._live),
                               _seed_slice(sc.critic.live_arena, K, 1, 2, sc.critic._live))
    finally:
        lib.sgrl_deterministic(prev)


def _buffers(K, n, rows):
    from sgrl_b200.buffer import ReplayBuffer
    bufs = []
    for k in range(K):
        buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=rows)
        b = synth.make_batch(rows, n, seed=60 + k)
        buf.add_batch(*(b[x].cuda() for x in ("obs", "action", "next_obs", "reward", "done")))
        bufs.append(buf)
    return bufs


def test_update_from_buffers_equals_update():
    """update_from_buffers == update on buf.get_batch of the same indices, bit for bit in deterministic mode; one library
    launch (the gather) outside the replayed graph per step."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    prev = lib.sgrl_deterministic(1)
    try:
        K, B, n = 3, 100, len(HUMANOID)
        g = G.build_graph(HUMANOID, device="cuda")
        bufs = _buffers(K, n, 400)
        a, b = SeedBatchedAgent(_args(), [7, 8, 9]), SeedBatchedAgent(_args(), [7, 8, 9])
        a.change_morphology(g); b.change_morphology(g)
        launches = []
        for it in range(7):
            random.seed(it)
            idx = [buf.draw_indices(B) for buf in bufs]
            la = a.update([buf.get_batch(ix) for buf, ix in zip(bufs, idx)], it)
            random.seed(it)
            l0 = lib.sgrl_launch_count()
            lb = b.update_from_buffers(bufs, B, it)
            launches.append(lib.sgrl_launch_count() - l0)
            for x, y in zip(la, lb):
                assert [float(v) for v in x.values()] == [float(v) for v in y.values()]
        torch.cuda.synchronize()
        for m in MODS:
            assert torch.equal(getattr(a, m).full_arena, getattr(b, m).full_arena), m
        assert launches[4:] == [1, 1, 1], launches       # its 0, 1: eager runs, 2, 3: captures of the two step kinds, then replays
        assert len(b._plans) == 1
    finally:
        lib.sgrl_deterministic(prev)


def test_update_from_buffers_errors():
    from sgrl_b200.buffer import ReplayBuffer
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), [1, 2])
    sb.change_morphology(G.build_graph(HUMANOID, device="cuda"))
    n = len(HUMANOID)
    bufs = _buffers(2, n, 50)
    with pytest.raises(ValueError, match="one per seed"):
        sb.update_from_buffers(bufs[:1], 10, 0)
    with pytest.raises(ValueError, match="do not match"):
        sb.update_from_buffers([bufs[0], _buffers(1, 5, 50)[0]], 10, 0)
    with pytest.raises(ValueError, match="empty"):
        sb.update_from_buffers([bufs[0], ReplayBuffer(41 * n, 3 * n, max_buffer_size=10)], 10, 0)
    with pytest.raises(ValueError, match="one per seed"):
        sb.update([_batch(10, n, 1)], 0)


@pytest.mark.parametrize("use_tc", [1, 0])
def test_select_actions_match_each_seed(use_tc):
    K = 3
    sb, singles = _agents([31, 32, 33], use_tc)
    graphs = [G.build_graph(p, device="cuda") for p in (HUMANOID, [-1, 0], CHAIN15, HUMANOID)]
    obs = [[synth.make_obs(1, len(g["parents"]), seed=10 * k + i).reshape(-1).numpy() for i, g in enumerate(graphs)] for k in range(K)]
    for rep in range(3):                                   # eager run, capture, replay
        got = sb.select_actions(obs, graphs)
        for k in range(K):
            want = singles[k].select_actions(obs[k], graphs)
            for x, y in zip(got[k], want):
                assert x.shape == y.shape
                err = np.linalg.norm(x - y) / max(np.linalg.norm(y), 1e-12)
                assert err <= TOL, (rep, k, err)


def test_launches_do_not_grow_with_seeds():
    """Library launches of one eager seed-batched step (with the actor step) at K = 1 and at K = 8."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    B, n = 100, len(HUMANOID)
    g = G.build_graph(HUMANOID, device="cuda")
    counts = {}
    for K in (1, 8):
        sb = SeedBatchedAgent(_args(), list(range(K)))
        sb.use_graphs = False
        sb.change_morphology(g)
        batches = [_batch(B, n, k) for k in range(K)]
        sb.update(batches, 0)                                  # first call: one-time set-up inside the library
        torch.cuda.synchronize()
        l0 = lib.sgrl_launch_count()
        sb.update(batches, 2)
        counts[K] = lib.sgrl_launch_count() - l0
    assert counts[8] <= counts[1], counts
