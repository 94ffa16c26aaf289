"""Per-seed TD3 hyper-parameters on the GPU.  The kernels that read the per-seed table (grouped Adam + clip, per-net Polyak,
critic loss, target-policy smoothing) against torch with distinct values per seed; seed-batched agents whose seeds all train
with different values against standalone Agents built with those values, on both GEMM paths; identical values changing
nothing bit for bit; no leaks between seeds; and values changed after the step's graphs were captured reaching the replayed
step, for SeedBatchedAgent.set_hparams and for a plain Agent's attributes."""
import random

import numpy as np
import pytest
import torch

from oracle import ref_loader
from sgrl_b200 import graph as G, morphologies as M, synth
from sgrl_b200._lib import CRITIC, TD3_HPARAMS, check, lib, ptr, stream
from test_seed_batch_gpu import HUMANOID, MODS, _batch, _compare_seed, _compare_seed_arenas, _noise, _seed_slice

pytestmark = pytest.mark.gpu

# every field differs between the seeds; seed 1 does not clip
HP = [dict(actor_lr=2e-4, critic_lr=3e-4, discount=0.97, policy_noise=0.3, noise_clip=0.4, grad_clipping_value=0.2,
           target_smoothing_tau=0.01, reward_scale=2.0),
      dict(actor_lr=5e-5, critic_lr=1e-4, discount=0.9, policy_noise=0.1, noise_clip=0.15, grad_clipping_value=0.0,
           target_smoothing_tau=0.05, reward_scale=0.5),
      dict(actor_lr=1e-4, critic_lr=5e-5, discount=0.995, policy_noise=0.2, noise_clip=0.05, grad_clipping_value=1.0,
           target_smoothing_tau=0.002, reward_scale=1.5)]


def _args():
    return ref_loader.default_args()


def _table(rows):
    """{field: value} per seed -> the device table (K SgrlTd3Hparams rows)."""
    t = np.zeros(len(rows), dtype=TD3_HPARAMS)
    for k, r in enumerate(rows):
        for f, v in r.items():
            t[f][k] = v
        t["one_minus_tau"][k] = 1.0 - float(np.float32(r.get("tau", 0.0)))
    return torch.from_numpy(t.view(np.uint8).copy()).cuda()


def _single(seed, h, use_tc):
    """The Agent seed k of a SeedBatchedAgent(args, seeds, hparams) must follow: seed's initial weights, h's values."""
    from sgrl_b200.agent import Agent
    from sgrl_b200.seed_batch import args_with
    torch.manual_seed(seed)
    ag = Agent(args_with(_args(), {**_base(), **h}))
    ag.actor_optimizer.lr, ag.critic_optimizer.lr = h.get("actor_lr", _args().lr), h.get("critic_lr", _args().lr)
    for m in MODS:
        getattr(ag, m).use_tc = use_tc
    return ag


def _base():
    from sgrl_b200.seed_batch import args_hparams
    return args_hparams(_args())


def _sweep(seeds, hps, use_tc):
    from sgrl_b200.seed_batch import SeedBatchedAgent
    sb = SeedBatchedAgent(_args(), seeds, hparams=hps)
    for m in MODS:
        getattr(sb, m).use_tc = use_tc
    return sb, [_single(s, h, use_tc) for s, h in zip(seeds, hps)]


def _rand(n, seed, scale=1.0):
    return torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)) * scale


# ---------------------------------------------------------------------------------------------------------- kernels

def test_grouped_adam_clip_matches_torch_per_seed():
    """K = 3 seeds of a twin-critic-shaped arena (nets k and K + k form seed k's group): each group against torch.optim.Adam with
    its own lr and clip_grad_norm_ with its own threshold (seed 1 unclipped), five steps, test_k6_gpu's tolerances."""
    K, n_net = 3, 50_000
    lrs, clips = (1e-4, 3e-4, 5e-5), (0.1, 0.0, 2.0)
    b1, b2, eps = 0.9, 0.999, 1e-8
    p = _rand(2 * K * n_net, 1)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    hi, lo = torch.empty_like(p), torch.empty_like(p)
    step = torch.zeros(1, dtype=torch.int32, device="cuda")
    ss = torch.zeros(2 * K, device="cuda")
    hp = _table([dict(critic_lr=lr, actor_lr=1.0, max_norm=c) for lr, c in zip(lrs, clips)])
    nets = lambda t, k: torch.cat([t[k * n_net:(k + 1) * n_net], t[(K + k) * n_net:(K + k + 1) * n_net]])
    refs = [torch.nn.Parameter(nets(p, k).clone()) for k in range(K)]
    opts = [torch.optim.Adam([r], lr=lr, betas=(b1, b2), eps=eps) for r, lr in zip(refs, lrs)]
    for it in range(5):
        g = _rand(p.numel(), 10 + it, 1.0 if it % 2 else 1e-3)
        for k in range(K):
            refs[k].grad = nets(g, k).clone()
            if clips[k] > 0:
                torch.nn.utils.clip_grad_norm_([refs[k]], clips[k])
            opts[k].step()
        ss.zero_()
        check(lib.sgrl_sumsq_nets(ptr(g), n_net, 2 * K, ptr(ss), stream()))
        check(lib.sgrl_bump_step(ptr(step), stream()))
        check(lib.sgrl_adam_clip_groups_hp(ptr(p), ptr(g), ptr(m), ptr(v), n_net, 2 * K, K, ptr(ss), ptr(step), ptr(hp), CRITIC, b1, b2, eps,
                                           1.0, ptr(hi), ptr(lo), stream()))
        for k in range(K):
            st = opts[k].state[refs[k]]
            got = nets(p, k)
            assert (got - refs[k].data).abs().max().item() <= 2e-7 * lrs[k] / 1e-4 + 1.2e-7 * got.abs().max().item(), (it, k)
            assert ((nets(m, k) - st["exp_avg"]).norm() / st["exp_avg"].norm()).item() < 1e-6, (it, k)
            assert ((nets(v, k) - st["exp_avg_sq"]).norm() / st["exp_avg_sq"].norm()).item() < 1e-6, (it, k)
    assert torch.equal(hi, ((p.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32))


def test_grouped_adam_with_one_table_row_is_the_by_value_kernel():
    n = 40_000
    g = _rand(n, 3)
    outs = []
    for use_table in (True, False):
        p, m, v = _rand(n, 2), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
        step = torch.ones(1, dtype=torch.int32, device="cuda")
        ss = (g.double() ** 2).sum().float().reshape(1)
        if use_table:
            check(lib.sgrl_adam_clip_groups_hp(ptr(p), ptr(g), ptr(m), ptr(v), n, 1, 1, ptr(ss), ptr(step), ptr(_table([dict(actor_lr=3e-4, max_norm=0.1)])),
                                               0, 0.9, 0.999, 1e-8, 0.5, None, None, stream()))
        else:
            check(lib.sgrl_adam_clip(ptr(p), ptr(g), ptr(m), ptr(v), n, ptr(ss), ptr(step), 3e-4, 0.9, 0.999, 1e-8, 0.1, 0.5, None, None, stream()))
        outs.append((p, m, v))
    assert all(torch.equal(x, y) for x, y in zip(*outs))


def test_per_net_polyak_is_bit_exact_per_seed():
    """K = 3 seeds, 6 nets ([live nets | dead nets]): net z, live or dead, follows tau*s + (1-tau)*t with seed z % K's tau."""
    K, nets, L, D = 3, 6, 6400, 1280
    taus = (0.005, 0.3, 1.0)
    n = nets * (L + D)
    s, t = _rand(n, 4), _rand(n, 5)
    want = t.clone()
    for z in range(nets):
        tau = taus[z % K]
        for a, b in ((z * L, (z + 1) * L), (nets * L + z * D, nets * L + (z + 1) * D)):
            want[a:b] = tau * s[a:b] + (1 - tau) * t[a:b]
    hi, lo = torch.zeros(nets * L, device="cuda"), torch.zeros(nets * L, device="cuda")
    check(lib.sgrl_polyak_hp(ptr(t), ptr(s), nets, L, D, ptr(_table([dict(tau=x) for x in taus])), K, ptr(hi), ptr(lo), stream()))
    assert torch.equal(t, want)
    rna = lambda x: ((x.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)
    assert torch.equal(hi, rna(t[:nets * L])) and torch.equal(lo, rna(t[:nets * L] - hi))


def test_critic_loss_takes_each_seeds_discount_and_reward_scale():
    K, Gr, N = 3, 60, 7
    T = Gr * N
    gen = torch.Generator(device="cuda").manual_seed(3)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    q, tq, rew = r(2 * K, T), r(2 * K, T), r(K, Gr) * 3 + 1
    done = (torch.rand(K, Gr, device="cuda", generator=gen) < 0.2).float()
    tokg = torch.arange(Gr, dtype=torch.int32, device="cuda").repeat_interleave(N).contiguous()
    disc, scale = (0.97, 0.9, 0.995), (2.0, 0.5, 1.5)
    hp = _table([dict(discount=d, reward_scale=s) for d, s in zip(disc, scale)])

    def run(fn, *scalars):
        target, dq, loss = torch.empty(K, T, device="cuda"), torch.empty(2 * K, T, device="cuda"), torch.zeros(K, device="cuda")
        st = torch.zeros(K, 2, dtype=torch.float64, device="cuda")
        check(fn(ptr(q), ptr(tq), ptr(rew), ptr(done), ptr(tokg), None, ptr(target), ptr(dq), ptr(loss), *scalars, T, ptr(st), Gr, K, stream()))
        return target, dq, loss, st

    target, dq, loss, st = run(lib.sgrl_td3_critic_loss_seeds_hp, ptr(hp))
    for k in range(K):
        rs = rew[k] * scale[k]
        y = rs[tokg.long()] + (1 - done[k][tokg.long()]) * disc[k] * torch.minimum(tq[k], tq[K + k])
        e1, e2 = q[k] - y, q[K + k] - y
        assert ((target[k] - y).abs().max() / y.abs().max()).item() < 1e-6, k
        assert ((dq[k] - 2 * e1 / T).abs().max() / (2 * e1 / T).abs().max()).item() < 1e-5, k
        assert ((dq[K + k] - 2 * e2 / T).abs().max() / (2 * e2 / T).abs().max()).item() < 1e-5, k
        want = ((e1.double() ** 2).sum() + (e2.double() ** 2).sum()).item() / T
        assert abs(loss[k].item() - want) <= 1e-5 * want, k
        assert abs(st[k, 0].item() - rs.double().sum().item()) <= 1e-9 * rs.double().abs().sum().item(), k
        assert abs(st[k, 1].item() - (rs.double() ** 2).sum().item()) <= 1e-9 * (rs.double() ** 2).sum().item(), k
        # the by-value kernel with seed k's scalars computes the same bits for seed k
        t2, d2, _, s2 = run(lib.sgrl_td3_critic_loss_seeds, disc[k], scale[k])
        assert torch.equal(t2[k], target[k]) and torch.equal(d2[k], dq[k]) and torch.equal(d2[K + k], dq[K + k]) and torch.equal(s2[k], st[k])


def test_smoothing_noise_per_seed():
    """In-kernel noise: each seed's noise_out has the standard deviation of its own sigma (>= 1e5 draws per seed), next_action is
    the clip of each seed's own noise_clip; equal rows draw what the by-value kernel draws over the whole batch; K = 1 is
    sgrl_td3_smooth_action_rng bit for bit.  The injected-noise kernel clips each seed by its own noise_clip."""
    K, T, amax, seed = 3, 34_000, 0.6, 0x1234_5678_9ABC
    per = 3 * T
    n = K * per
    sig, clip = (0.3, 0.1, 0.2), (0.4, 0.15, 0.05)
    a = _rand(n, 7, 0.3)
    draw = torch.full((1,), 5, dtype=torch.int32, device="cuda")
    out, nz = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    check(lib.sgrl_td3_smooth_action_rng_hp(ptr(a), ptr(out), ptr(nz), ptr(_table([dict(policy_noise=s, noise_clip=c) for s, c in zip(sig, clip)])),
                                            per, amax, n, seed, ptr(draw), stream()))
    for k in range(K):
        sl = slice(k * per, (k + 1) * per)
        assert abs(nz[sl].double().std().item() / sig[k] - 1) < 0.02, k
        c = torch.tensor(clip[k], dtype=torch.float32, device="cuda")
        assert torch.equal(out[sl], torch.clamp(a[sl] + torch.maximum(torch.minimum(nz[sl], c), -c), -amax, amax)), k
        inside = a[sl].abs() < amax - clip[k]                   # where max_action does not clamp, the move is at most the clip
        assert ((out[sl] - a[sl])[inside].abs() <= clip[k] * (1 + 1e-6)).all() and ((nz[sl].abs() > clip[k]) & inside).any(), k
    # equal rows: the draws are the by-value kernel's over the whole batch
    o1, n1, o2, n2 = (torch.empty(n, device="cuda") for _ in range(4))
    check(lib.sgrl_td3_smooth_action_rng_hp(ptr(a), ptr(o1), ptr(n1), ptr(_table([dict(policy_noise=0.2, noise_clip=0.5)] * K)), per, amax, n, seed,
                                            ptr(draw), stream()))
    check(lib.sgrl_td3_smooth_action_rng(ptr(a), ptr(o2), ptr(n2), 0.2, 0.5, amax, n, seed, ptr(draw), stream()))
    assert torch.equal(o1, o2) and torch.equal(n1, n2)
    # K = 1
    o1, n1, o2, n2 = (torch.empty(per, device="cuda") for _ in range(4))
    check(lib.sgrl_td3_smooth_action_rng_hp(ptr(a), ptr(o1), ptr(n1), ptr(_table([dict(policy_noise=0.3, noise_clip=0.4)])), per, amax, per, seed,
                                            ptr(draw), stream()))
    check(lib.sgrl_td3_smooth_action_rng(ptr(a), ptr(o2), ptr(n2), 0.3, 0.4, amax, per, seed, ptr(draw), stream()))
    assert torch.equal(o1, o2) and torch.equal(n1, n2)
    # injected noise
    noise = _rand(n, 8, 0.3)
    out = torch.empty(n, device="cuda")
    check(lib.sgrl_td3_smooth_action_hp(ptr(a), ptr(noise), ptr(out), ptr(_table([dict(noise_clip=c) for c in clip])), per, amax, n, stream()))
    for k in range(K):
        sl = slice(k * per, (k + 1) * per)
        c = torch.tensor(clip[k], dtype=torch.float32, device="cuda")
        assert torch.equal(out[sl], torch.clamp(a[sl] + torch.maximum(torch.minimum(noise[sl], c), -c), -amax, amax)), k
        ref = torch.empty(per, device="cuda")
        check(lib.sgrl_td3_smooth_action(ptr(a[sl]), ptr(noise[sl]), ptr(ref), clip[k], amax, per, stream()))
        assert torch.equal(out[sl], ref), k


# ---------------------------------------------------------------------------------------------------------- whole steps

def _check_losses(got, want, tol, what):
    assert set(got) == set(want)
    for key in want:
        a, b = float(got[key]), float(want[key])
        assert abs(a - b) <= tol * max(abs(b), 1e-6), f"{what} {key}: {a} vs {b}"


@pytest.mark.parametrize("use_tc", [1, 0])
@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
def test_seeds_follow_agents_built_with_their_values(graphs, use_tc):
    """K = 3, every per-seed value different, four updates with injected noise: each seed against an Agent built with its
    values, at the tolerances of test_seed_batch_gpu.test_seeds_follow_their_own_agents."""
    K, B, n = 3, 100, len(HUMANOID)
    sb, singles = _sweep([21, 22, 23], HP, use_tc)
    g = G.build_graph(HUMANOID, device="cuda")
    for ag in [sb] + singles:
        ag.use_graphs = graphs
        ag.change_morphology(g)
    what = f"graphs={graphs} use_tc={use_tc}"
    for it in range(4):
        batches = [_batch(B, n, 100 * k + it) for k in range(K)]
        noises = [_noise(B, n, 1000 * k + it) for k in range(K)]
        got = sb.update(batches, it, noises)
        for k in range(K):
            _check_losses(got[k], singles[k].update(batches[k], it, noise=noises[k]), 1e-5 if it == 0 else 1e-4, f"{what} it {it} seed {k}")
        if it == 0:
            torch.cuda.synchronize()
            for k in range(K):
                _compare_seed(sb, k, singles[k], what + " after the first update")
    torch.cuda.synchronize()
    for k in range(K):
        _compare_seed_arenas(sb, k, singles[k], what + " after four updates")


@pytest.mark.parametrize("use_tc", [1, 0])
def test_packed_seeds_follow_agents_built_with_their_values(use_tc):
    """The same through update_packed_per_seed on three hopper morphologies against Agent.update_packed."""
    K = 3
    names, sizes = ["3d_hopper_3_shin", "3d_hopper_4_lower_shin", "3d_hopper_5_full"], (24, 16, 20)
    gs = [G.build_graph(M.ALL[x], device="cuda") for x in names]
    sb, singles = _sweep([31, 32, 33], HP, use_tc)
    for it in range(4):
        batches = [[(g, _batch(B, len(g["parents"]), 1000 * k + 10 * i + it)) for i, (g, B) in enumerate(zip(gs, sizes))] for k in range(K)]
        noises = [[_noise(B, len(g["parents"]), 5000 + 1000 * k + 10 * i + it) for i, (g, B) in enumerate(zip(gs, sizes))] for k in range(K)]
        got = sb.update_packed_per_seed(batches, it, noises)
        for k in range(K):
            _check_losses(got[k], singles[k].update_packed(batches[k], it, noises[k]), 1e-5 if it == 0 else 1e-4, f"packed it {it} seed {k}")
    torch.cuda.synchronize()
    for k in range(K):
        _compare_seed_arenas(sb, k, singles[k], f"packed use_tc={use_tc} after four updates")


def _run(sb, it0, n_it, B=100):
    n = len(HUMANOID)
    out = []
    for it in range(it0, it0 + n_it):
        out.append(sb.update([_batch(B, n, 10 * it + k) for k in range(sb.n_seeds)], it))
    torch.cuda.synchronize()
    return out


def _state(ag):
    return [getattr(ag, m).full_arena.clone() for m in MODS]


def test_identical_values_change_nothing():
    """Deterministic mode: explicit hparams equal to args are bit-identical to none; K = 1 with non-default values is the Agent
    built with them bit for bit, with the same launches."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    prev = lib.sgrl_deterministic(1)
    try:
        g = G.build_graph(HUMANOID, device="cuda")
        runs = []
        for hps in (None, [dict(_base()) for _ in range(3)], [{"lr": _args().lr}] * 3):
            sb = SeedBatchedAgent(_args(), [1, 2, 3], hparams=hps)
            sb.change_morphology(g)
            runs.append((_run(sb, 0, 4), _state(sb)))
        for losses, state in runs[1:]:
            assert [[float(v) for v in d.values()] for l in losses for d in l] == [[float(v) for v in d.values()] for l in runs[0][0] for d in l]
            assert all(torch.equal(x, y) for x, y in zip(state, runs[0][1]))
        sb, (ag,) = _sweep([5], [HP[1]], 1)
        sb.change_morphology(g); ag.change_morphology(g)
        n, counts = len(HUMANOID), {"sb": [], "ag": []}
        for it in range(6):
            b = _batch(100, n, 300 + it)
            l0 = lib.sgrl_launch_count()
            got = sb.update([b], it)[0]                         # noise drawn in the kernel: the plans' Philox seeds agree
            counts["sb"].append(lib.sgrl_launch_count() - l0)
            l0 = lib.sgrl_launch_count()
            want = ag.update(b, it)
            counts["ag"].append(lib.sgrl_launch_count() - l0)
            assert [float(got[k]) for k in want] == [float(want[k]) for k in want], it
        torch.cuda.synchronize()
        assert counts["sb"] == counts["ag"]
        psb, pag = next(iter(sb._plans.values())), next(iter(ag._plans.values()))
        assert psb.graph_launches == pag.graph_launches and psb.graph_launches
        assert all(torch.equal(x, y) for x, y in zip(_state(sb), _state(ag)))
    finally:
        lib.sgrl_deterministic(prev)


def test_changing_one_seed_does_not_leak():
    """Deterministic mode: other values for seed 1 only leave seeds 0 and 2 bit-identical; seed 1 differs."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    prev = lib.sgrl_deterministic(1)
    try:
        K = 3
        g = G.build_graph(HUMANOID, device="cuda")
        res = []
        for hps in (HP, [HP[0], HP[2], HP[2]]):
            sb = SeedBatchedAgent(_args(), [1, 2, 3], hparams=hps)
            sb.change_morphology(g)
            res.append((sb, _run(sb, 0, 4)))
        (sa, la), (sc, lc) = res
        for k in (0, 2):
            for m in MODS:
                mod = getattr(sa, m)
                per = mod._nb // K
                assert torch.equal(_seed_slice(mod.live_arena, K, k, per, mod._live), _seed_slice(getattr(sc, m).live_arena, K, k, per, mod._live)), (m, k)
            assert [float(v) for l in la for v in l[k].values()] == [float(v) for l in lc for v in l[k].values()], k
        assert not torch.equal(_seed_slice(sa.critic.live_arena, K, 1, 2, sa.critic._live), _seed_slice(sc.critic.live_arena, K, 1, 2, sc.critic._live))
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


def test_set_hparams_after_capture_reaches_the_replayed_step():
    """Four updates from the buffers, then set_hparams on seeds 1 and 2 (seed 2's clip from 0 to 0.1) and four more: each seed
    matches its own Agent changed at the same step.  Nothing is recaptured (the plan and its graph keys stay; each replayed
    step makes one library launch, the gather, outside the graph).  Deterministic mode: in the default mode seed 0's critic
    drifts from its Agent by up to 7e-5 over these eight updates in some runs and by 1e-8 in others, from the second update
    on and without any set_hparams (two runs of the batched agent alone differ as much; measured on a B200), which would hide
    a wrong value as well as flag a right one.  With the mode on, both sides are reproducible and every seed stays within
    TOL (worst 6.5e-6, seed 0)."""
    prev = lib.sgrl_deterministic(1)
    try:
        _set_hparams_after_capture()
    finally:
        lib.sgrl_deterministic(prev)


def _set_hparams_after_capture():
    K, B, n = 3, 100, len(HUMANOID)
    hps = [HP[0], HP[1], {**HP[2], "grad_clipping_value": 0.0}]
    sb, singles = _sweep([7, 8, 9], hps, 1)
    g = G.build_graph(HUMANOID, device="cuda")
    for ag in [sb] + singles:
        ag.change_morphology(g)
    bufs = _buffers(K, n, 400)
    change = {1: dict(lr=2e-4, discount=0.95, noise_clip=0.3, target_smoothing_tau=0.02, reward_scale=3.0),
              2: dict(critic_lr=1e-4, grad_clipping_value=0.1, policy_noise=0.25, target_smoothing_tau=0.01)}
    launches, keys = [], None
    for it in range(8):
        if it == 4:
            plan = next(iter(sb._plans.values()))
            keys = (id(plan), set(plan.graphs))
            for k, ch in change.items():
                sb.set_hparams(k, **ch)
                one = singles[k]
                one.actor_optimizer.lr = ch.get("actor_lr", ch.get("lr", one.actor_optimizer.lr))
                one.critic_optimizer.lr = ch.get("critic_lr", ch.get("lr", one.critic_optimizer.lr))
                for key in ("discount", "noise_clip", "policy_noise", "grad_clipping_value"):
                    if key in ch:
                        one.args[key] = ch[key]
                one.target_smoothing_tau = ch.get("target_smoothing_tau", one.target_smoothing_tau)
                one.reward_scale = ch.get("reward_scale", one.reward_scale)
                assert sb.get_hparams(k) == one._seed_hparams()[0]
        noises = [_noise(B, n, 1000 * k + it) for k in range(K)]
        random.seed(it)
        l0 = lib.sgrl_launch_count()
        got = sb.update_from_buffers(bufs, B, it, noises)
        launches.append(lib.sgrl_launch_count() - l0)
        random.seed(it)
        for k in range(K):
            _check_losses(got[k], singles[k].update_from_buffer(bufs[k], B, it, noise=noises[k]), 1e-5 if it == 0 else 1e-4, f"it {it} seed {k}")
    torch.cuda.synchronize()
    for k in range(K):
        _compare_seed_arenas(sb, k, singles[k], "after the change")
    plan = next(iter(sb._plans.values()))
    assert len(sb._plans) == 1 and (id(plan), set(plan.graphs)) == keys == (keys[0], {(True, False), (False, False)})
    assert launches[4:] == [1, 1, 1, 1], launches


def test_agent_attributes_changed_after_capture_reach_the_replayed_step():
    """A plain Agent: critic_optimizer.lr, target_smoothing_tau, reward_scale and args.discount set after the step's graphs were
    captured.  The replaying agent equals an eager one started from the same state every step, at the tolerances of
    test_agent_gpu's graph-against-eager race test, and its reward statistics use the new reward_scale."""
    from sgrl_b200.agent import Agent
    torch.manual_seed(4)
    ag = Agent(_args())
    torch.manual_seed(4)
    eg = Agent(_args())
    eg.use_graphs = False
    g = G.build_graph(HUMANOID, device="cuda")
    ag.change_morphology(g); eg.change_morphology(g)
    B, n = 100, len(HUMANOID)
    rel = lambda a, b: ((a.double() - b.double()).norm() / b.double().norm()).item()
    for it in range(8):
        if it == 5:
            for x in (ag, eg):
                x.critic_optimizer.lr, x.target_smoothing_tau, x.reward_scale = 1e-3, 0.05, 2.5
                x.args.discount = 0.9
        eg.load_state_dict(ag.state_dict())
        eg.critic_optimizer.load_state_dict(ag.critic_optimizer.state_dict())
        eg.actor_optimizer.load_state_dict(ag.actor_optimizer.state_dict())
        b = _batch(B, n, 50 + it)
        noise = _noise(B, n, 100 + it)
        la, le = ag.update(b, it, noise=noise), eg.update(b, it, noise=noise)
        assert abs(la["loss/critic_loss"].item() - le["loss/critic_loss"].item()) <= 1e-6 * abs(le["loss/critic_loss"].item()), it
        want_mean = (b["reward"].double() * ag.reward_scale).mean().item()
        assert abs(la["misc/train_reward_mean"] - want_mean) <= 1e-6 * max(abs(want_mean), 1e-2), it
        assert rel(ag.critic.grad_arena(), eg.critic.grad_arena()) < 1e-5, it
        for m in MODS:
            assert rel(getattr(ag, m).full_arena, getattr(eg, m).full_arena) < 1e-5, (it, m)
    assert set(next(iter(ag._plans.values())).graphs) == {(True, False), (False, False)}
