"""Seed-batched packed multi-morphology updates on the GPU (SeedBatchedAgent.update_packed_per_seed /
update_packed_from_buffers_per_seed, sgrl_b200.buffer.gather_seeds_into, sgrl_replay_gather_seeds): the K x M-buffer gather is
bit-exact against per-buffer get_batch; each seed follows its own Agent.update_packed on both GEMM paths, in graph and eager
mode; K = 1 is Agent.update_packed bit for bit; seeds do not leak into each other; the buffer path equals the batch path and
draws what K agents draw; one plan, one launch outside the replayed graph; K = 8 seeds x the 23 CWHH morphologies; and an end
to end loop of acting, storing transitions and updating."""
import random
import warnings

import numpy as np
import pytest
import torch

from sgrl_b200 import graph as G, morphologies as M, synth
from sgrl_b200._lib import ReplayPart, lib, ptr, stream
from test_seed_batch_gpu import MODS, _agents, _args, _batch, _compare_seed, _compare_seed_arenas, _noise, _seed_slice

pytestmark = pytest.mark.gpu

MIX = ["3d_hopper_5_full", "3d_humanoid_9_full", "3d_cheetah_14_full", "3d_walker_7_full"]
SIZES = (24, 16, 12, 20)
CWHH = sorted(M.SETS["3d_cwhh"])
KEYS = ("obs", "action", "next_obs", "reward", "done")


def _graphs(names):
    return [G.build_graph(M.ALL[n], device="cuda") for n in names]


def _seed_batches(graphs, sizes, K, it):
    return [[(g, _batch(B, len(g["parents"]), 1000 * k + 10 * i + it)) for i, (g, B) in enumerate(zip(graphs, sizes))] for k in range(K)]


def _seed_noises(graphs, sizes, K, it):
    return [[_noise(B, len(g["parents"]), 5000 + 1000 * k + 10 * i + it) for i, (g, B) in enumerate(zip(graphs, sizes))] for k in range(K)]


def _add_rows(buf, n, seed, host=False):
    """n synthetic transitions: host-side add_transition (left staged until the next flush) or one device add_batch."""
    b = synth.make_batch(n, buf.obs_dim // 41, seed=seed)
    if host:
        for i in range(n):
            buf.add_transition(b["obs"][i].numpy(), b["action"][i].numpy(), b["next_obs"][i].numpy(), float(b["reward"][i]),
                               float(b["done"][i]))
    else:
        buf.add_batch(*(b[k].cuda() for k in KEYS))


def _mix_buffers(seed):
    """One seed's buffers of MIX: the 5-limb one wrapped, the 9-limb one holding fewer rows than a batch, the 14-limb one with
    unflushed add_transition rows on top of device rows, the 7-limb one part full.  Every seed fills the same row counts."""
    from sgrl_b200.buffer import ReplayBuffer
    n = [len(M.ALL[m]) for m in MIX]
    bufs = [ReplayBuffer(41 * k, 3 * k, max_buffer_size=cap) for k, cap in zip(n, (64, 1000, 500, 300))]
    for i in range(4):
        _add_rows(bufs[0], 40, seed=100 * seed + 1 + i)
    _add_rows(bufs[1], 20, seed=100 * seed + 5)
    _add_rows(bufs[2], 200, seed=100 * seed + 6)
    _add_rows(bufs[2], 37, seed=100 * seed + 7, host=True)
    _add_rows(bufs[3], 250, seed=100 * seed + 8)
    return bufs


def _mix_parts(K):
    graphs = _graphs(MIX)
    return [list(zip(graphs, _mix_buffers(k))) for k in range(K)]


def _expected(bufs, indices):
    """The packed batch by torch indexing of each buffer's rows (negative indices wrap as in numpy), split into its columns:
    independent of the library's gather."""
    cols = {k: [] for k in KEYS}
    for b, ix in zip(bufs, indices):
        b.flush()
        r = b.rows[torch.as_tensor(ix, dtype=torch.int64, device=b.rows.device)]
        od, ad = b.obs_dim, b.action_dim
        for k, x in zip(KEYS, (r[:, :od], r[:, od:od + ad], r[:, od + ad:2 * od + ad], r[:, -2], r[:, -1])):
            cols[k].append(x.reshape(-1))
    return {k: torch.cat(v) for k, v in cols.items()}


def _nan_outputs(bufs, counts):
    f = lambda n: torch.full((n,), float("nan"), device="cuda")
    return (f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(c * b.action_dim for c, b in zip(counts, bufs))),
            f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(counts)), f(sum(counts)))


def _cwhh_buffers(K):
    """K seeds x the 23 CWHH morphologies: buffer i wrapped (i % 3 == 0), part full (1) or with unflushed host rows on top of
    device rows (2); capacities differ per morphology, row counts are the same for every seed."""
    from sgrl_b200.buffer import ReplayBuffer
    out = []
    for k in range(K):
        bufs = []
        for i, name in enumerate(CWHH):
            n, cap = len(M.ALL[name]), 16 + 3 * i
            buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=cap)
            if i % 3 == 0:
                _add_rows(buf, cap, seed=1000 * k + i)
                _add_rows(buf, cap // 2 + 3, seed=1000 * k + i + 500)
            elif i % 3 == 1:
                _add_rows(buf, cap // 2, seed=1000 * k + i)
            else:
                _add_rows(buf, cap // 2, seed=1000 * k + i)
                _add_rows(buf, 3, seed=1000 * k + i + 500, host=True)
            bufs.append(buf)
        out.append(bufs)
    return out


def test_gather_over_seeds_is_bit_exact():
    from sgrl_b200.buffer import gather_seeds_into
    K = 8
    seeds = _cwhh_buffers(K)
    assert seeds[3][2]._staged > 0                                      # rows the gather must flush first
    counts = [3 + i % 4 for i in range(len(CWHH))]
    idx = [[np.random.default_rng(100 * k + i).integers(-b.max_buffer_size, b.max_buffer_size, c).tolist()
            for i, (b, c) in enumerate(zip(bufs, counts))] for k, bufs in enumerate(seeds)]
    assert any(x < 0 for ixs in idx for ix in ixs for x in ix)
    flat_bufs = [b for bufs in seeds for b in bufs]
    flat_idx = [ix for ixs in idx for ix in ixs]
    out = _nan_outputs(flat_bufs, counts * K)
    l0 = lib.sgrl_launch_count()
    assert gather_seeds_into(seeds, idx, *out) == sum(counts) * K
    assert lib.sgrl_launch_count() - l0 == 1
    want = _expected(flat_bufs, flat_idx)
    for k, got in zip(KEYS, out):
        assert torch.equal(got, want[k]), k
    # the full 8 x 64 = 512 descriptors (buffers may repeat)
    wide = [(bufs * 3)[:64] for bufs in seeds]
    wide_idx = [(ixs * 3)[:64] for ixs in idx]
    wide_counts = (counts * 3)[:64]
    out = _nan_outputs([b for bufs in wide for b in bufs], wide_counts * K)
    gather_seeds_into(wide, wide_idx, *out)
    want = _expected([b for bufs in wide for b in bufs], [ix for ixs in wide_idx for ix in ixs])
    for k, got in zip(KEYS, out):
        assert torch.equal(got, want[k]), k
    # refused in Python before anything is launched ...
    l0 = lib.sgrl_launch_count()
    with pytest.raises(ValueError, match="1 to 8 seeds"):
        gather_seeds_into(seeds + seeds[:1], idx + idx[:1], *_nan_outputs(flat_bufs + seeds[0], counts * (K + 1)))
    with pytest.raises(ValueError, match="1 to 64 buffers"):
        gather_seeds_into([bufs * 3 for bufs in seeds[:2]], [ixs * 3 for ixs in idx[:2]], *_nan_outputs(flat_bufs * 3, counts * 6))
    assert lib.sgrl_launch_count() == l0
    # ... and by the library itself
    b0 = seeds[0][0]
    desc = (ReplayPart * 130)()
    for d in desc:
        d.rows, d.row_floats, d.capacity, d.obs_dim, d.act_dim, d.batch = ptr(b0.rows), b0.row_floats, b0.max_buffer_size, b0.obs_dim, b0.action_dim, 1
    dev_idx = torch.zeros(130, dtype=torch.int64, device="cuda")
    o = [ptr(t) for t in out]

    def call(n_parts, n_seeds):
        return lib.sgrl_replay_gather_seeds(desc, n_parts, n_seeds, ptr(dev_idx), *o, stream())

    assert call(9, 9) < 0 and b"n_seeds must be 1..8" in lib.sgrl_last_error()
    assert call(130, 2) < 0 and b"n_parts must be" in lib.sgrl_last_error()          # 65 parts per seed
    assert call(5, 2) < 0 and b"n_parts must be" in lib.sgrl_last_error()
    desc[23].batch = 2                                                               # seed 1's part 3 of 20 per seed
    assert call(60, 3) < 0 and b"seed 1 part 3" in lib.sgrl_last_error()
    desc[23].batch, desc[23].obs_dim = 1, b0.obs_dim + 41
    assert call(60, 3) < 0 and b"seed 1 part 3" in lib.sgrl_last_error()
    assert lib.sgrl_launch_count() == l0


@pytest.mark.parametrize("use_tc", [1, 0])
@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
def test_seeds_follow_their_own_agents(graphs, use_tc):
    """K = 3 on hopper-5 / humanoid-9 / cheetah-14 / walker-7, four updates, each seed against its own Agent.update_packed:
    the tolerances of test_seed_batch_gpu.test_seeds_follow_their_own_agents."""
    K = 3
    sb, singles = _agents([21, 22, 23], use_tc)
    gs = _graphs(MIX)
    for ag in [sb] + singles:
        ag.use_graphs = graphs
    what = f"packed graphs={graphs} use_tc={use_tc}"
    for it in range(4):
        batches, noises = _seed_batches(gs, SIZES, K, it), _seed_noises(gs, SIZES, K, it)
        got = sb.update_packed_per_seed(batches, it, noises)
        assert len(got) == K
        for k in range(K):
            want = singles[k].update_packed(batches[k], it, noises[k])
            assert set(got[k]) == set(want)
            for key in want:
                a, b = float(got[k][key]), float(want[key])
                tol = 1e-5 if it == 0 else 1e-4
                assert abs(a - b) <= tol * max(abs(b), 1e-6), f"{what} it {it} seed {k} {key}: {a} vs {b}"
        if it == 0:
            torch.cuda.synchronize()
            for k in range(K):
                _compare_seed(sb, k, singles[k], what + " after the first update")
    torch.cuda.synchronize()
    for k in range(K):
        _compare_seed_arenas(sb, k, singles[k], what + " after four updates")


@pytest.mark.parametrize("use_tc", [1, 0])
def test_one_seed_is_update_packed_bit_for_bit(use_tc):
    prev = lib.sgrl_deterministic(1)
    try:
        sb, (ag,) = _agents([5], use_tc)
        gs = _graphs(MIX)
        counts = {"sb": [], "ag": []}
        for it in range(6):
            b, nz = _seed_batches(gs, SIZES, 1, it)[0], _seed_noises(gs, SIZES, 1, it)[0]
            l0 = lib.sgrl_launch_count()
            got = sb.update_packed_per_seed([b], it, [nz])[0]
            counts["sb"].append(lib.sgrl_launch_count() - l0)
            l0 = lib.sgrl_launch_count()
            want = ag.update_packed(b, it, nz)
            counts["ag"].append(lib.sgrl_launch_count() - l0)
            assert set(got) == set(want)
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
    """K = 3 in deterministic mode: two runs are bit-identical, and another batch of one morphology for seed 1 leaves seeds 0
    and 2 bit-identical."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    prev = lib.sgrl_deterministic(1)
    try:
        K = 3
        gs = _graphs(MIX)
        data = [_seed_batches(gs, SIZES, K, it) for it in range(4)]
        noise = [_seed_noises(gs, SIZES, K, it) for it in range(4)]
        runs = []
        for variant in range(3):
            sb = SeedBatchedAgent(_args(), [1, 2, 3])
            d = [[list(p) for p in x] for x in data]
            if variant == 2:
                for it in range(4):
                    d[it][1][2] = (gs[2], _batch(SIZES[2], len(gs[2]["parents"]), 777 + it))
            losses = [sb.update_packed_per_seed(d[it], it, noise[it]) for it in range(4)]
            torch.cuda.synchronize()
            runs.append((sb, losses))
        (sa, la), (sb_, lb), (sc, lc) = runs
        for m in MODS:
            assert torch.equal(getattr(sa, m).full_arena, getattr(sb_, m).full_arena), m
        for m in ("actor", "critic"):
            assert torch.equal(getattr(sa, m).grad_arena(), getattr(sb_, m).grad_arena()), m
        assert [[float(v) for d in l for v in d.values()] for l in la] == [[float(v) for d in l for v in d.values()] for l in lb]
        for k in (0, 2):
            for m in MODS:
                x, y = getattr(sa, m), getattr(sc, m)
                assert torch.equal(_seed_slice(x.live_arena, K, k, x._nb // K, x._live), _seed_slice(y.live_arena, K, k, y._nb // K, y._live)), (m, k)
            for it in range(4):
                assert float(la[it][k]["loss/critic_loss"]) == float(lc[it][k]["loss/critic_loss"])
        assert not torch.equal(_seed_slice(sa.critic.live_arena, K, 1, 2, sa.critic._live), _seed_slice(sc.critic.live_arena, K, 1, 2, sc.critic._live))
    finally:
        lib.sgrl_deterministic(prev)


@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
def test_buffer_path_equals_sampled_batches(graphs):
    """update_packed_from_buffers_per_seed == update_packed_per_seed of buf.sample batches drawn in the same order, bit for
    bit in deterministic mode, leaving the same Python random state."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    prev = lib.sgrl_deterministic(1)
    try:
        K, B = 3, 32
        parts = _mix_parts(K)
        a, b = SeedBatchedAgent(_args(), [7, 8, 9]), SeedBatchedAgent(_args(), [7, 8, 9])
        a.use_graphs = b.use_graphs = graphs
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)                 # the 9-limb buffers hold fewer rows than B
            for it, s in enumerate((11, 12, 13, 14, 15, 16)):
                random.seed(s)
                la = a.update_packed_from_buffers_per_seed(parts, B, it)
                st = random.getstate()
                random.seed(s)
                lb = b.update_packed_per_seed([[(g, buf.sample(B)) for g, buf in p] for p in parts], it)
                assert random.getstate() == st
                for x, y in zip(la, lb):
                    assert x.keys() == y.keys()
                    assert [float(v) for v in x.values()] == [float(v) for v in y.values()], it
        torch.cuda.synchronize()
        for m in MODS:
            assert torch.equal(getattr(a, m).full_arena, getattr(b, m).full_arena), m
    finally:
        lib.sgrl_deterministic(prev)


@pytest.mark.parametrize("allow_duplicate", [False, True])
def test_draws_are_those_of_agents_in_seed_order(allow_duplicate):
    """The rows a seed-batched step draws (Python's random or numpy's stream) are the rows K agents calling
    update_packed_from_buffers one after the other in seed order draw."""
    K, B = 2, 16
    sb, singles = _agents([3, 4], 1)
    parts = _mix_parts(K)
    drawn = []
    for p in parts:
        for _, buf in p:
            def rec(*a, _f=buf.draw_indices, **kw):
                ix = _f(*a, **kw)
                drawn.append(list(np.asarray(ix)))
                return ix
            buf.draw_indices = rec
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        random.seed(9); np.random.seed(9)
        sb.update_packed_from_buffers_per_seed(parts, B, 0, allow_duplicate=allow_duplicate)
        mine, drawn[:] = list(drawn), []
        st = (random.getstate(), np.random.get_state()[1].tobytes())
        random.seed(9); np.random.seed(9)
        for k in range(K):
            singles[k].update_packed_from_buffers(parts[k], B, 0, allow_duplicate=allow_duplicate)
    assert mine == drawn and len(mine) == K * len(MIX)
    assert (random.getstate(), np.random.get_state()[1].tobytes()) == st


def test_one_plan_one_launch_and_launches_do_not_grow():
    """Both methods share one plan; a replayed step makes one library launch outside the graph (the gather); below
    the grouped-projection size (32 768 tokens x nets, run_group in csrc/net.cuh) the captured graphs hold as many library
    launches for K = 4 as for K = 1."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    B, plans = 32, {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for K in (4, 1):
            sb = SeedBatchedAgent(_args(), list(range(K)))
            parts = _mix_parts(K)
            for it in range(4):                                          # eager run + capture of both step kinds
                sb.update_packed_from_buffers_per_seed(parts, B, it)
            assert len(sb._plans) == 1 and len(sb._packed_tables) == 1
            plan = next(iter(sb._plans.values()))
            assert len(plan.graphs) == 2
            assert 2 * K * plan.tb.T <= 32768                            # grouped launches (csrc/net.cuh run_group) for both K
            graphs = dict(plan.graphs)
            for it in range(4, 8):
                sb.update_packed_per_seed([[(g, buf.sample(B)) for g, buf in p] for p in parts], it)
                assert len(sb._plans) == 1 and len(sb._packed_tables) == 1
            for it in range(8, 12):
                l0 = lib.sgrl_launch_count()
                sb.update_packed_from_buffers_per_seed(parts, B, it)
                assert lib.sgrl_launch_count() - l0 == 1, it
            assert plan.graphs == graphs and next(iter(sb._plans.values())) is plan
            plans[K] = dict(plan.graph_launches)
    assert plans[4] == plans[1] and all(plans[1].values()), plans


def test_eight_seeds_on_cwhh():
    """K = 8 seeds x the 23 CWHH morphologies x B = 8: nb = 16 critic nets over ragged tables and the 184-part gather.  Seeds
    0 and 7 match their own Agents after one update."""
    K, B = 8, 8
    sb, singles = _agents(list(range(K)), 1)
    seeds = _cwhh_buffers(K)
    gs = _graphs(CWHH)
    parts = [list(zip(gs, bufs)) for bufs in seeds]
    rows = [min(B, buf.max_sample_size) for buf in seeds[0]]
    noises = _seed_noises(gs, rows, K, 0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        random.seed(3)
        got = sb.update_packed_from_buffers_per_seed(parts, B, 0, noises)
        random.seed(3)
        want = {}
        for k in range(K):
            if k in (0, K - 1):
                want[k] = singles[k].update_packed_from_buffers(parts[k], B, 0, noises[k])
            else:
                for buf in seeds[k]:
                    buf.draw_indices(B)
    assert sb.critic._nb == 16 and len(next(iter(sb._plans.values())).tb.parts) == len(CWHH)
    torch.cuda.synchronize()
    for k, w in want.items():
        for key in w:
            a, b = float(got[k][key]), float(w[key])
            assert abs(a - b) <= 1e-5 * max(abs(b), 1e-6), (k, key, a, b)
        _compare_seed(sb, k, singles[k], f"CWHH K=8 seed {k}")


def test_end_to_end_acting_storing_updating():
    """K = 2 seeds x 3 morphologies x 2 envs each, four iterations of select_actions -> add_transition ->
    update_packed_from_buffers_per_seed, each seed against its own Agent doing select_actions -> add_transition ->
    update_packed_from_buffers on its own buffers."""
    from sgrl_b200.buffer import ReplayBuffer
    K, B, names = 2, 4, ["3d_hopper_5_full", "3d_humanoid_9_full", "3d_walker_7_full"]
    sb, singles = _agents([41, 42], 1)
    gs = _graphs(names)
    env_graphs = [g for g in gs for _ in range(2)]
    nl = [len(g["parents"]) for g in env_graphs]

    def parts():
        return [(g, ReplayBuffer(41 * len(g["parents"]), 3 * len(g["parents"]), max_buffer_size=64)) for g in gs]

    sb_parts, ag_parts = [parts() for _ in range(K)], [parts() for _ in range(K)]
    start = [[synth.make_obs(1, n, seed=10 * k + e).reshape(-1).numpy().astype(np.float32) for e, n in enumerate(nl)] for k in range(K)]
    obs_sb, obs_ag = [list(o) for o in start], [list(o) for o in start]

    def step(obs, act, store):
        """A deterministic stand-in environment: next observation, reward and done from (obs, action)."""
        for e, (o, a) in enumerate(zip(obs, act)):
            a = a.reshape(-1)
            nxt = (0.9 * o + 0.1 * np.resize(a, o.shape)).astype(np.float32)
            store[e // 2][1].add_transition(o, a, nxt, float(np.tanh(a).sum() * 0.1), 0.0)
            obs[e] = nxt

    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)                     # the first batches are larger than the buffers
        for it in range(4):
            act_sb = sb.select_actions(obs_sb, env_graphs)
            for k in range(K):
                act_ag = singles[k].select_actions(obs_ag[k], env_graphs)
                step(obs_sb[k], act_sb[k], sb_parts[k])
                step(obs_ag[k], act_ag, ag_parts[k])
            rows = [min(B, 2 * (it + 1))] * len(gs)
            noises = _seed_noises(gs, rows, K, it)
            random.seed(500 + it)
            got = sb.update_packed_from_buffers_per_seed(sb_parts, B, it, noises)
            random.seed(500 + it)
            for k in range(K):
                want = singles[k].update_packed_from_buffers(ag_parts[k], B, it, noises[k])
                assert set(got[k]) == set(want)
                for key in want:
                    a, b = float(got[k][key]), float(want[key])
                    assert abs(a - b) <= 1e-4 * max(abs(b), 1e-6), (it, k, key, a, b)
            if it == 0:
                torch.cuda.synchronize()
                for k in range(K):
                    _compare_seed(sb, k, singles[k], "end to end, first update")
    torch.cuda.synchronize()
    for k in range(K):
        _compare_seed_arenas(sb, k, singles[k], "end to end, four iterations")


def test_cpu_buffers_are_refused():
    """A buffer whose rows live on the CPU is refused by update_packed_from_buffers_per_seed (the agent is on the GPU), before
    anything is drawn or a plan is created."""
    from sgrl_b200.buffer import ReplayBuffer
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), [1, 2])
    parts = _mix_parts(2)
    g, buf = parts[1][2]
    on_cpu = ReplayBuffer(buf.obs_dim, buf.action_dim, max_buffer_size=16, device="cpu")
    _add_rows(on_cpu, 4, seed=8, host=True)
    state = (random.getstate(), np.random.get_state()[1].tobytes())
    with pytest.raises(ValueError, match="seed 1 buffer 2 keeps its rows on cpu"):
        sb.update_packed_from_buffers_per_seed([parts[0], parts[1][:2] + [(g, on_cpu)] + parts[1][3:]], 8, 0)
    assert (random.getstate(), np.random.get_state()[1].tobytes()) == state
    assert len(sb._plans) == 0 and len(sb._packed_tables) == 0
