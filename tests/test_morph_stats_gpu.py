"""Per-morphology TD3 statistics of packed updates on the GPU (sgrl_td3_part_stats, the `per_morphology` keyword of
Agent.update_packed / update_packed_from_buffers and SeedBatchedAgent.update_packed_per_seed /
update_packed_from_buffers_per_seed).  The kernel against fp64 torch through the C ABI; each morphology's losses against the
fp64 oracle's per-morphology losses; the flag only observes (same parameters, Adam state and main dicts bit for bit, one
more launch, no recapture of the unflagged graphs); and every entry point, seed count, morph_count, lazy_stats and host or
device batches agreeing with each other."""
import contextlib
import random
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loader, set_oracle as O
from sgrl_b200._lib import check, lib, ptr, stream
from test_agent_gpu import make_agent
from test_packed_gpu import _parts
from test_seed_batch_gpu import MODS, _agents
from test_seed_hparams_gpu import _table
from test_seed_packed_gpu import CWHH, MIX, SIZES, _cwhh_buffers, _graphs, _mix_parts, _seed_batches, _seed_noises

pytestmark = pytest.mark.gpu

KEYS = ("loss/critic_loss", "misc/train_reward_mean", "misc/train_reward_var", "loss/actor_loss")


@contextlib.contextmanager
def _deterministic():
    prev = lib.sgrl_deterministic(1)
    try:
        yield
    finally:
        lib.sgrl_deterministic(prev)


def _floats(pm):
    """A per_morphology list as comparable tuples (NaN == NaN)."""
    return [tuple((k, repr(float(d[k]))) for k in d) for d in pm]


def _scale(pm, key):
    """Mean magnitude of one value over the morphologies: the scale a mean over them is compared at (actor losses of
    different signs may cancel)."""
    return sum(abs(float(d[key])) for d in pm) / len(pm)


# ------------------------------------------------------------------------------------------------------------ kernel

def _ragged(P):
    """P parts alternating 2-, 16-, 5- and 9-limb graphs with ragged batch sizes; the last part of several holds one sample."""
    parts, t0, g0 = [], 0, 0
    for i in range(P):
        n = (2, 16, 5, 9)[i % 4]
        B = 1 if (P > 1 and i == P - 1) else 1 + (7 * i + 3) % 13
        parts.append((t0, t0 + B * n, g0, g0 + B))
        t0, g0 = t0 + B * n, g0 + B
    return parts, t0, g0


@pytest.mark.parametrize("K", [1, 3, 8])
@pytest.mark.parametrize("P", [1, 4, 64])
def test_kernel_matches_fp64_torch(K, P):
    parts, T, Gr = _ragged(P)
    gen = torch.Generator(device="cuda").manual_seed(100 * K + P)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    q, target, q1 = r(2 * K, T), r(K, T), r(K, T) * 0.5 + 2.0          # positive offsets: the sums do not cancel
    reward = r(K, Gr) * 3 + 1
    scales = [0.5 + 0.75 * k for k in range(K)]
    hp = _table([dict(reward_scale=s, discount=0.9) for s in scales])
    table = torch.tensor(parts, dtype=torch.int32, device="cuda")

    def run(q1_):
        out = torch.full((K, P, 4), -1.0, dtype=torch.float64, device="cuda")
        check(lib.sgrl_td3_part_stats(ptr(q), ptr(target), ptr(q1_), ptr(reward), ptr(table), P, T, Gr, K, ptr(hp), ptr(out), stream()))
        torch.cuda.synchronize()
        return out

    got = run(q1)
    for k in range(K):
        for i, (t0, t1, g0, g1) in enumerate(parts):
            y = target[k, t0:t1].double()
            e1, e2 = q[k, t0:t1].double() - y, q[K + k, t0:t1].double() - y
            rs = (reward[k, g0:g1] * torch.tensor(scales[k], dtype=torch.float32, device="cuda")).double()
            want = [((e1 ** 2 + e2 ** 2).sum() / (t1 - t0)).item(), (-q1[k, t0:t1].double().sum() / (t1 - t0)).item(), rs.mean().item(),
                    rs.var().item() if g1 - g0 > 1 else float("nan")]
            for j, w in enumerate(want):
                g = got[k, i, j].item()
                if w != w:
                    assert g != g, (k, i, j, g)
                else:
                    assert abs(g - w) <= 1e-12 * abs(w), (k, i, j, g, w)
    if P > 1:
        assert torch.isnan(got[:, P - 1, 3]).all()                       # B_m = 1: no unbiased variance
    no_actor = run(None)
    assert torch.isnan(no_actor[..., 1]).all()
    idx = [0, 2, 3]
    assert torch.equal(no_actor[..., idx].nan_to_num(7.0), got[..., idx].nan_to_num(7.0))
    again = run(q1)
    assert torch.equal(again.view(torch.int64), got.view(torch.int64))      # bit for bit, NaN payloads included

    # refusals: negative code, a message, nothing launched, nothing written
    out = torch.full((K, P, 4), 7.0, dtype=torch.float64, device="cuda")
    n0 = lib.sgrl_launch_count()
    a = dict(q=ptr(q), target=ptr(target), q1=ptr(q1), reward=ptr(reward), parts=ptr(table), P=P, T=T, G=Gr, K=K, hp=ptr(hp))
    bad = [(dict(P=0), b"P must be"), (dict(P=65), b"P must be"), (dict(K=0), b"K must be"), (dict(K=9), b"K must be"),
           (dict(T=0), b"empty batch"), (dict(G=0), b"empty batch")]
    bad += [({name: None}, b"null pointer") for name in ("q", "target", "reward", "parts", "hp")]
    for kw, msg in bad:
        c = {**a, **kw}
        rc = lib.sgrl_td3_part_stats(c["q"], c["target"], c["q1"], c["reward"], c["parts"], c["P"], c["T"], c["G"], c["K"], c["hp"],
                                     ptr(out), stream())
        assert rc < 0 and msg in lib.sgrl_last_error(), (kw, rc, lib.sgrl_last_error())
    assert lib.sgrl_td3_part_stats(a["q"], a["target"], a["q1"], a["reward"], a["parts"], P, T, Gr, K, a["hp"], None, stream()) < 0
    torch.cuda.synchronize()
    assert lib.sgrl_launch_count() == n0
    assert torch.equal(out, torch.full_like(out, 7.0))


# ------------------------------------------------------------------------------------------------- against the oracle

def _oracle_packed_update_per_morphology(pa, pc, pa_t, pc_t, parts, it, opt_c, opt_a, lr=1e-4):
    """test_packed_gpu._oracle_packed_update, also returning each morphology's mse(q1,y) + mse(q2,y) and -Q1(obs, pi(obs)).mean()."""
    m = len(parts)
    loss_c, per_c = 0.0, []
    for g, b, nz in parts:
        with torch.no_grad():
            a2 = (O.actor_forward(pa_t, b["next_obs"], g) + nz.clamp(-0.5, 0.5)).clamp(-1.0, 1.0)
            tq1, tq2 = O.critic_forward(pc_t, b["next_obs"], a2, g)
            y = b["reward"] + (1 - b["done"]) * 0.99 * torch.min(tq1, tq2)
        q1, q2 = O.critic_forward(pc, b["obs"], b["action"], g)
        lm = F.mse_loss(q1, y) + F.mse_loss(q2, y)
        per_c.append(lm.item())
        loss_c = loss_c + lm / m
    opt_c.zero_grad()
    loss_c.backward()
    torch.nn.utils.clip_grad_norm_([p for p in pc.values() if p.requires_grad], 0.1)
    opt_c.step()
    out = {"critic": per_c}
    if it % 2 == 0:
        loss_a, per_a = 0.0, []
        for g, b, _ in parts:
            lm = -O.critic_forward(pc, b["obs"], O.actor_forward(pa, b["obs"], g), g, which=(1,)).mean()
            per_a.append(lm.item())
            loss_a = loss_a + lm / m
        opt_a.zero_grad()
        loss_a.backward()
        torch.nn.utils.clip_grad_norm_([p for p in pa.values() if p.requires_grad], 0.1)
        opt_a.step()
        out["actor"] = per_a
        with torch.no_grad():
            for src, dst in ((pc, pc_t), (pa, pa_t)):
                for k in src:
                    dst[k].mul_(1 - 0.005).add_(src[k].detach(), alpha=0.005)
    return out


@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
def test_per_morphology_matches_oracle(graphs):
    ag, pa0, pc0 = make_agent()
    ag.use_graphs = graphs
    parts = _parts()
    dd = torch.float64
    conv = lambda d, grad: {k: v.cuda().to(dd).requires_grad_(grad and not O.is_dead(k)) for k, v in d.items()}
    pa, pc, pa_t, pc_t = conv(pa0, True), conv(pc0, True), conv(pa0, False), conv(pc0, False)
    opt_c = torch.optim.Adam([p for p in pc.values() if p.requires_grad], lr=1e-4)
    opt_a = torch.optim.Adam([p for p in pa.values() if p.requires_grad], lr=1e-4)
    parts64 = []
    for g, b, nz in parts:
        g64 = dict(g); g64["relation"] = g["relation"].double()
        parts64.append((g64, {k: v.double() for k, v in b.items()}, nz.double()))
    scale = ag.reward_scale
    for it in range(4):
        ld = ag.update_packed([(g, b) for g, b, _ in parts], it, noises=[nz for _, _, nz in parts], per_morphology=True)
        ref = _oracle_packed_update_per_morphology(pa, pc, pa_t, pc_t, parts64, it, opt_c, opt_a)
        pm = ld["per_morphology"]
        assert len(pm) == len(parts)
        for i, (d, (_, b, _)) in enumerate(zip(pm, parts)):
            assert list(d) == [k for k in KEYS if it % 2 == 0 or k != "loss/actor_loss"]
            assert all(isinstance(v, float) for v in d.values())
            assert abs(d["loss/critic_loss"] - ref["critic"][i]) < 2e-4 * abs(ref["critic"][i]), (it, i, d, ref["critic"][i])
            if it % 2 == 0:
                assert abs(d["loss/actor_loss"] - ref["actor"][i]) < 5e-4 * abs(ref["actor"][i]), (it, i, d, ref["actor"][i])
            rs = (b["reward"].reshape(-1) * torch.tensor(scale, dtype=torch.float32, device="cuda")).double()
            assert abs(d["misc/train_reward_mean"] - rs.mean().item()) <= 1e-12 * rs.abs().mean().item()
            assert abs(d["misc/train_reward_var"] - rs.var().item()) <= 1e-12 * rs.var().item()
        for key, main in (("loss/critic_loss", "loss/critic_loss"),) + ((("loss/actor_loss", "loss/actor_loss"),) if it % 2 == 0 else ()):
            mean = sum(d[key] for d in pm) / len(pm)
            assert abs(mean - ld[main].item()) <= 1e-5 * _scale(pm, key), (it, key, mean, ld[main].item())


# ----------------------------------------------------------------------------------------------- the flag only observes

def _state(ag):
    out = {m: getattr(ag, m).full_arena.clone() for m in MODS}
    for name in ("actor_optimizer", "critic_optimizer"):
        opt = getattr(ag, name)
        out.update({name + ".m": opt.exp_avg.clone(), name + ".v": opt.exp_avg_sq.clone(), name + ".step": opt.step_count.clone()})
    return out


def test_flag_only_observes():
    """Deterministic mode, six steps (steps 2..5 replayed from captured graphs): an agent that asks for the statistics on every
    step ends bit-identical to one that never does, with the same main dicts."""
    parts = _parts()
    with _deterministic():
        (a, _, _), (b, _, _) = make_agent(), make_agent()
        la, lb = [], []
        for it in range(6):
            batches, noises = [(g, x) for g, x, _ in parts], [nz for _, _, nz in parts]
            la.append(a.update_packed(batches, it, noises, per_morphology=True))
            lb.append(b.update_packed(batches, it, noises))
        torch.cuda.synchronize()
        sa, sb = _state(a), _state(b)
        for k in sa:
            assert torch.equal(sa[k], sb[k]), k
        for x, y in zip(la, lb):
            assert set(x) - set(y) == {"per_morphology"}
            assert all(float(x[k]) == float(y[k]) for k in y)
        pa, pb = next(iter(a._plans.values())), next(iter(b._plans.values()))
        assert set(pa.graphs) == {(True, False, True), (False, False, True)} and set(pb.graphs) == {(True, False), (False, False)}
        for (s, r, _), n in pa.graph_launches.items():
            assert n == pb.graph_launches[(s, r)] + 1


def test_flagged_graphs_beside_unflagged_ones():
    """One plan: the flagged graphs hold exactly one more library launch than the unflagged ones, and alternating the flag
    keeps replaying the same four CUDAGraph objects (nothing recaptured)."""
    ag, _, _ = make_agent()
    parts = _parts()
    batches, noises = [(g, x) for g, x, _ in parts], [nz for _, _, nz in parts]
    for it in range(8):                                                  # eager run + capture of each of the four graphs
        ag.update_packed(batches, it, noises, per_morphology=it >= 4)
    plan = next(iter(ag._plans.values()))
    assert len(plan.graphs) == 4
    for s in (True, False):
        assert plan.graph_launches[(s, False, True)] == plan.graph_launches[(s, False)] + 1
    held = dict(plan.graphs)
    for it in range(8, 16):
        on = (it // 2) % 2 == 0
        l0 = lib.sgrl_launch_count()
        ld = ag.update_packed(batches, it, noises, per_morphology=on)
        assert lib.sgrl_launch_count() == l0                             # replayed: no launch outside the graph
        assert ("per_morphology" in ld) == on
    assert len(plan.graphs) == 4 and all(plan.graphs[k] is g for k, g in held.items())
    assert next(iter(ag._plans.values())) is plan


# --------------------------------------------------------------------------------------- every path agrees with the others

def test_buffer_path_equals_batch_path():
    from sgrl_b200.agent import Agent
    with _deterministic(), warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)                     # a buffer holding fewer rows than a batch
        parts = _mix_parts(1)[0]
        torch.manual_seed(4); a = Agent(ref_loader.default_args())
        torch.manual_seed(4); b = Agent(ref_loader.default_args())
        for it, s in enumerate((1, 2, 3, 4)):
            random.seed(s)
            la = a.update_packed_from_buffers(parts, 32, it, per_morphology=True)
            random.seed(s)
            lb = b.update_packed([(g, buf.sample(32)) for g, buf in parts], it, per_morphology=True)
            assert _floats(la["per_morphology"]) == _floats(lb["per_morphology"]), it


HP4 = [dict(reward_scale=s, discount=d) for s, d in ((1.0, 0.99), (2.5, 0.9), (0.25, 0.97), (4.0, 0.995))]


def _close(got, want, tol, what):
    """Within tol relative, or 1e-7 absolute: an actor loss near zero is the mean of Q-values of order 0.1..1, whose fp32
    reassociation between K nets and one net moves it by about 1e-8."""
    assert [list(d) for d in got] == [list(d) for d in want], what
    for i, (x, y) in enumerate(zip(got, want)):
        for key in y:
            a, b = float(x[key]), float(y[key])
            assert abs(a - b) <= max(tol * abs(b), 1e-7), (what, i, key, a, b)


@pytest.mark.parametrize("path", ["batches", "buffers"])
def test_seeds_equal_their_agents(path):
    """K = 4 seeds with their own reward_scale and discount: seed k's list is agent(k)'s, two steps (actor and critic-only)."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    K = 4
    sb = SeedBatchedAgent(ref_loader.default_args(), [11, 12, 13, 14], hparams=HP4)
    singles = [sb.agent(k) for k in range(K)]
    gs = _graphs(MIX)
    mix = _mix_parts(K)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for it in range(2):
            if path == "batches":
                batches, noises = _seed_batches(gs, SIZES, K, it), _seed_noises(gs, SIZES, K, it)
                got = sb.update_packed_per_seed(batches, it, noises, per_morphology=True)
                want = [singles[k].update_packed(batches[k], it, noises[k], per_morphology=True) for k in range(K)]
            else:
                random.seed(20 + it); np.random.seed(20 + it)
                got = sb.update_packed_from_buffers_per_seed(mix, 24, it, per_morphology=True)
                random.seed(20 + it); np.random.seed(20 + it)
                want = [singles[k].update_packed_from_buffers(mix[k], 24, it, per_morphology=True) for k in range(K)]
            for k in range(K):
                # K nets and one net sum Q in different orders; one morphology's loss over a few dozen samples does not
                # average that out the way the mean over morphologies does (1.5e-5 seen on a 20-sample part)
                _close(got[k]["per_morphology"], want[k]["per_morphology"], 1e-4, f"{path} it {it} seed {k}")
                for x, y in zip(got[k]["per_morphology"], want[k]["per_morphology"]):   # same rewards, same scale: same bits
                    assert repr(x["misc/train_reward_mean"]) == repr(y["misc/train_reward_mean"])
                    assert repr(x["misc/train_reward_var"]) == repr(y["misc/train_reward_var"])


@pytest.mark.parametrize("use_tc", [1, 0])
def test_one_seed_is_an_agent_bit_for_bit(use_tc):
    with _deterministic():
        sb, (ag,) = _agents([5], use_tc)
        gs = _graphs(MIX)
        for it in range(4):
            b, nz = _seed_batches(gs, SIZES, 1, it)[0], _seed_noises(gs, SIZES, 1, it)[0]
            got = sb.update_packed_per_seed([b], it, [nz], per_morphology=True)[0]
            want = ag.update_packed(b, it, nz, per_morphology=True)
            assert _floats(got["per_morphology"]) == _floats(want["per_morphology"]), it


def test_eight_seeds_on_cwhh():
    """K = 8 seeds x the 23 CWHH morphologies (184 CTAs): the means over morphologies are the main dicts' losses, and the reward
    statistics are those of the rows the step gathered."""
    from sgrl_b200.seed_batch import SeedBatchedAgent
    K, B = 8, 8
    sb = SeedBatchedAgent(ref_loader.default_args(), list(range(K)), hparams=[dict(reward_scale=0.5 + k) for k in range(K)])
    gs = _graphs(CWHH)
    parts = [list(zip(gs, bufs)) for bufs in _cwhh_buffers(K)]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for it in range(2):
            got = sb.update_packed_from_buffers_per_seed(parts, B, it, per_morphology=True)
            plan = next(iter(sb._plans.values()))
            rew = plan.rew.view(K, -1).clone()
            for k in range(K):
                pm = got[k]["per_morphology"]
                assert len(pm) == len(CWHH)
                keys = ("loss/critic_loss", "loss/actor_loss") if it == 0 else ("loss/critic_loss",)
                for key in keys:
                    mean = sum(d[key] for d in pm) / len(pm)
                    assert abs(mean - got[k][key].item()) <= 1e-5 * _scale(pm, key), (it, k, key, mean, got[k][key].item())
                scale = torch.tensor(0.5 + k, dtype=torch.float32, device="cuda")
                for d, (_, _, g0, g1, _) in zip(pm, plan.tb.parts):
                    rs = (rew[k, g0:g1] * scale).double()
                    assert abs(d["misc/train_reward_mean"] - rs.mean().item()) <= 1e-12 * max(rs.abs().mean().item(), 1e-12)
                    if g1 - g0 > 1:
                        assert abs(d["misc/train_reward_var"] - rs.var().item()) <= 1e-12 * max(rs.var().item(), 1e-12)


def test_morph_count_leaves_per_morphology_values_unchanged():
    """morph_count = 2 M scales the main dict's losses by M / morph_count and leaves the per-morphology values alone: a
    critic-only step from the same state gives the same bits; on an actor step (whose actor loss reads a critic stepped on the
    rescaled gradient) the per-morphology means are the main losses times morph_count / M."""
    parts = _parts()
    M_ = len(parts)
    batches, noises = [(g, x) for g, x, _ in parts], [nz for _, _, nz in parts]
    with _deterministic():
        for it in (1, 0):
            (a, _, _), (b, _, _) = make_agent(), make_agent()
            la = a.update_packed(batches, it, noises, per_morphology=True)
            lb = b.update_packed(batches, it, noises, morph_count=2 * M_, per_morphology=True)
            assert abs(lb["loss/critic_loss"].item() - la["loss/critic_loss"].item() / 2) <= 1e-6 * la["loss/critic_loss"].item()
            for x, y in zip(la["per_morphology"], lb["per_morphology"]):
                assert list(x) == list(y)
                for key in x:
                    if key != "loss/actor_loss":
                        assert repr(x[key]) == repr(y[key]), (it, key)
            for key in ("loss/critic_loss", "loss/actor_loss") if it == 0 else ("loss/critic_loss",):
                mean = sum(d[key] for d in lb["per_morphology"]) / M_
                assert abs(mean / 2 - lb[key].item()) <= 1e-5 * _scale(lb["per_morphology"], key) / 2, (it, key, mean, lb[key].item())


def test_lazy_host_and_deterministic_runs_agree():
    """Deterministic mode: host batches with floats, device batches with lazy 0-dim fp64 device tensors and a second run of
    the host batches all give the same bits."""
    parts = _parts()
    runs = []
    with _deterministic():
        for variant in ("host", "lazy", "host"):
            ag, _, _ = make_agent()
            ag.lazy_stats = variant == "lazy"
            out = []
            for it in range(3):
                if variant == "host":
                    batches = [(g, {k: v.cpu() for k, v in x.items()}) for g, x, _ in parts]
                else:
                    batches = [(g, x) for g, x, _ in parts]
                ld = ag.update_packed(batches, it, [nz for _, _, nz in parts], per_morphology=True)
                for d in ld["per_morphology"]:
                    for v in d.values():
                        if variant == "lazy":
                            assert torch.is_tensor(v) and v.is_cuda and v.dtype == torch.float64 and v.dim() == 0
                        else:
                            assert isinstance(v, float)
                out.append(_floats(ld["per_morphology"]))
            runs.append(out)
    assert runs[0] == runs[1] == runs[2]
