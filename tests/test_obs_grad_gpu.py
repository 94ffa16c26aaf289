"""Gradient w.r.t. the observation input through SEPolicy / SECritic (loss.backward() reaches `state`), against the fp64
autograd of the oracle; its rotation behaviour (the gradient of an invariant loss rotates with the limb vectors about gravity);
ragged packed tables through backward_raw(dobs=); and that requesting it changes nothing else (deterministic mode: same
parameter gradients and d/d(action) bit for bit, one extra launch)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import set_oracle as O
from sgrl_b200 import _lib, graph as G, morphologies as M, synth
from sgrl_b200.modules import make_packed_tables
import gpu_util
import parity
from test_backward_gpu import grad_report, oracle_grads
from test_parity_wide_gpu import Verdict, _traces

pytestmark = pytest.mark.gpu

CASES = [(n, B) for n, B in parity.CASES[:4]] + [("3d_humanoid_9_full", 100), ("3d_humanoid_9_full", 256)]
IDS = [f"{n}-B{B}" for n, B in CASES]


@pytest.fixture(scope="module", params=[1, 0], ids=["tcgen05", "simt"])
def mods(request):
    return gpu_util.make_modules(use_tc=request.param)


@pytest.fixture(scope="module")
def gold():
    return parity.load_golden()


def _case(gold, name, B):
    """golden batches for parity.CASES, synthetic (seed 1) for the larger humanoid batches"""
    par = M.ALL[name]
    if (name, B) in parity.CASES:
        return parity.golden_graph(gold, name, par, device="cuda"), parity.golden_batch(gold, name, device="cuda")
    return G.build_graph(par, device="cuda"), gpu_util.to_cuda(synth.make_batch(B, len(par), seed=1))


def _g64(g):
    g64 = dict(g); g64["relation"] = g["relation"].double()
    return g64


def _p64(params):
    return {k: v.cuda().double() for k, v in params.items()}


def _oracle_input_grads(loss_fn, *inputs):
    """fp64 gradients of loss_fn(*inputs) w.r.t. every input"""
    xs = [x.detach().double().requires_grad_(True) for x in inputs]
    loss = loss_fn(*xs)
    return torch.autograd.grad(loss, xs)


def _assert_param_grads(name, B, what, got, params, loss_fn, flips_and_masks):
    """The parameter gradients of the same backward, held to the bounds the suite already uses: on the golden batches 1e-4 of
    the fp64 oracle on every tensor (tests/test_backward_gpu.py); on the synthetic humanoid batches the same, or a miss fully
    explained by relu units on their kink (tests/test_parity_wide_gpu.py, Verdict): every unit the CUDA forward puts on the
    other side of zero sits within 1e-5 of its row's scale, and the oracle run with the CUDA activation pattern agrees to 1e-4.
    loss_fn(p, masks) is the fp64 loss (masks None: the oracle's own activations); flips_and_masks() -> (flips, masks)."""
    _, want = oracle_grads(params, lambda p: loss_fn(p, None))
    v = Verdict(what, *grad_report(got, want))
    if (name, B) in parity.CASES:
        assert v.ok, str(v)
        return
    if not v.ok:
        flips, masks = flips_and_masks()
        v.flips += flips
        _, want2 = oracle_grads(params, lambda p: loss_fn(p, masks))
        v.bad_forced, v.glob_forced = grad_report(got, want2)
    assert v.ok or v.explained, str(v)


def _actor_flips_and_masks(actor, pa, b, g64, B, N):
    tb = actor._tables(B)
    _, st_a = actor.forward_raw(tb, b["obs"].contiguous(), None, keep=True, nb=1)
    torch.cuda.synchronize()
    tr = _traces(_p64(pa), ("actor.",), b["obs"].view(B, N, 41).double(), g64)["actor."]
    return gpu_util.relu_flips(actor, st_a, tb, 1, 0, tr, "actor."), gpu_util.relu_masks(actor, st_a, tb, 1, 0)


@pytest.mark.parametrize("name,B", CASES, ids=IDS)
def test_critic_td_loss_state_gradient(mods, gold, name, B):
    _, critic, _, pc = mods
    g, b = _case(gold, name, B)
    critic.change_morphology(g)
    critic.zero_grad(set_to_none=True)
    s = b["obs"].clone().requires_grad_(True)
    a = b["action"].clone().requires_grad_(True)
    q1, q2 = critic(s, a)
    tgt = b["reward"].expand_as(q1)
    (F.mse_loss(q1, tgt) + F.mse_loss(q2, tgt)).backward()
    pc64, g64 = _p64(pc), _g64(g)

    def lf(p, s_, a_, masks=None):
        o1, o2 = O.critic_forward(p, s_, a_, g64, masks=masks)
        t = b["reward"].double().expand_as(o1)
        return F.mse_loss(o1, t) + F.mse_loss(o2, t)
    ds, da = _oracle_input_grads(lambda s_, a_: lf(pc64, s_, a_), b["obs"], b["action"])
    assert s.grad is not None and s.grad.shape == s.shape
    assert parity.rel_err(s.grad, ds) < parity.RTOL
    assert parity.rel_err(a.grad, da) < parity.RTOL

    def flips_and_masks():
        N = len(g["parents"])
        tb = critic._tables(B)
        _, stash = critic.forward_raw(tb, b["obs"].contiguous(), b["action"].contiguous(), keep=True)
        torch.cuda.synchronize()
        x = torch.cat([b["obs"].view(B, N, 41), b["action"].view(B, N, 3)], 2).double()
        tr = _traces(pc64, ("critic1.", "critic2."), x, g64)
        flips, masks = [], {}
        for z, pre in enumerate(("critic1.", "critic2.")):
            flips += gpu_util.relu_flips(critic, stash, tb, 2, z, tr[pre], pre)
            masks[z + 1] = gpu_util.relu_masks(critic, stash, tb, 2, z)
        return flips, masks
    got = {k: p.grad for k, p in critic.named_parameters()}
    _assert_param_grads(name, B, "critic", got, pc, lambda p, mk: lf(p, b["obs"].double(), b["action"].double(), mk), flips_and_masks)


@pytest.mark.parametrize("name,B", CASES, ids=IDS)
def test_critic_q1_state_gradient(mods, gold, name, B):
    _, critic, _, pc = mods
    g, b = _case(gold, name, B)
    critic.change_morphology(g)
    critic.zero_grad(set_to_none=True)
    s = b["obs"].clone().requires_grad_(True)
    a = b["action"].clone().requires_grad_(True)
    critic.Q1(s, a).mean().backward()
    pc64, g64 = _p64(pc), _g64(g)
    ds, da = _oracle_input_grads(lambda s_, a_: O.critic_forward(pc64, s_, a_, g64, which=(1,)).mean(), b["obs"], b["action"])
    assert parity.rel_err(s.grad, ds) < parity.RTOL
    assert parity.rel_err(a.grad, da) < parity.RTOL
    assert all(p.grad is None for k, p in critic.named_parameters() if k.startswith("critic2."))


@pytest.mark.parametrize("name,B", CASES, ids=IDS)
def test_actor_state_gradient(mods, gold, name, B):
    actor, _, pa, _ = mods
    g, b = _case(gold, name, B)
    actor.change_morphology(g)
    actor.zero_grad(set_to_none=True)
    c = torch.randn(b["action"].shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64).cuda()
    s = b["obs"].clone().requires_grad_(True)
    (actor(s) * c.float()).sum().backward()
    pa64, g64 = _p64(pa), _g64(g)
    (ds,) = _oracle_input_grads(lambda s_: (O.actor_forward(pa64, s_, g64) * c).sum(), b["obs"])
    assert parity.rel_err(s.grad, ds) < parity.RTOL
    got = {k: p.grad for k, p in actor.named_parameters()}
    _assert_param_grads(name, B, "actor", got, pa, lambda p, mk: (O.actor_forward(p, b["obs"].double(), g64, masks=mk) * c).sum(),
                        lambda: _actor_flips_and_masks(actor, pa, b, g64, B, len(g["parents"])))


@pytest.mark.parametrize("name,B", CASES, ids=IDS)
def test_actor_loss_chain_state_gradient(mods, gold, name, B):
    """-Q1(s, actor(s)).mean(): the state gradient arrives through both modules and is summed by autograd"""
    actor, critic, pa, pc = mods
    g, b = _case(gold, name, B)
    actor.change_morphology(g); critic.change_morphology(g)
    actor.zero_grad(set_to_none=True); critic.zero_grad(set_to_none=True)
    s = b["obs"].clone().requires_grad_(True)
    (-critic.Q1(s, actor(s)).mean()).backward()
    pa64, pc64, g64 = _p64(pa), _p64(pc), _g64(g)
    (ds,) = _oracle_input_grads(lambda s_: -O.critic_forward(pc64, s_, O.actor_forward(pa64, s_, g64), g64, which=(1,)).mean(), b["obs"])
    assert parity.rel_err(s.grad, ds) < parity.RTOL
    N = len(g["parents"])

    def lf(p, mk):
        mk_a, mk_c = mk if mk is not None else (None, None)
        a = O.actor_forward(p, b["obs"].double(), g64, masks=mk_a)
        return -O.critic_forward(pc64, b["obs"].double(), a, g64, which=(1,), masks=None if mk_c is None else {1: mk_c}).mean()

    def flips_and_masks():
        flips, mk_a = _actor_flips_and_masks(actor, pa, b, g64, B, N)
        tb = actor._tables(B)
        a_out, _ = actor.forward_raw(tb, b["obs"].contiguous(), None, keep=True, nb=1)
        _, st_c = critic.forward_raw(tb, b["obs"].contiguous(), a_out[0].contiguous(), keep=True, nb=1)
        torch.cuda.synchronize()
        with torch.no_grad():
            a_ref = O.actor_forward(pa64, b["obs"].double(), g64)
        xc = torch.cat([b["obs"].view(B, N, 41).double(), a_ref.view(B, N, 3)], 2)
        flips += gpu_util.relu_flips(critic, st_c, tb, 1, 0, _traces(pc64, ("critic1.",), xc, g64)["critic1."], "critic1.")
        return flips, (mk_a, gpu_util.relu_masks(critic, st_c, tb, 1, 0))
    got = {k: p.grad for k, p in actor.named_parameters()}
    _assert_param_grads(name, B, "actor", got, pa, lf, flips_and_masks)


# ---------------------------------------------------------------------------------------------------------------- subequivariance
def _rotate_grad(grad, n, angle):
    """rotate_about_gravity acts on the 8 limb vectors (columns 0..23); the gradient of an invariant loss transforms the same way"""
    return synth.rotate_about_gravity(grad, n, angle)


@pytest.mark.parametrize("which", ["critic", "actor"])
def test_state_gradient_rotates_with_the_limb_vectors(mods, which):
    actor, critic, _, _ = mods
    name, B, angle = "3d_humanoid_9_full", 100, 0.7
    par = M.ALL[name]
    n = len(par)
    g = G.build_graph(par, device="cuda")
    b = gpu_util.to_cuda(synth.make_batch(B, n, seed=1))
    actor.change_morphology(g); critic.change_morphology(g)

    def grad_at(obs):
        s = obs.clone().requires_grad_(True)
        if which == "critic":
            q1, q2 = critic(s, b["action"])
            tgt = b["reward"].expand_as(q1)
            loss = F.mse_loss(q1, tgt) + F.mse_loss(q2, tgt)
        else:
            loss = actor(s).pow(2).sum()
        loss.backward()
        return s.grad
    g0 = grad_at(b["obs"])
    gr = grad_at(synth.rotate_about_gravity(b["obs"], n, angle))
    want = _rotate_grad(g0, n, angle)
    assert parity.rel_err(gr, want) < parity.RTOL
    # the scalar part (columns 24..40 of each limb) is invariant, the vector part is not (the check above is not vacuous)
    assert parity.rel_err(gr.view(B, n, 41)[..., 24:], g0.view(B, n, 41)[..., 24:]) < parity.RTOL
    assert parity.rel_err(gr.view(B, n, 41)[..., :24], g0.view(B, n, 41)[..., :24]) > 1e-2


# ---------------------------------------------------------------------------------------------------------------- ragged packed tables
PACKED = [([-1, 0], 5), (M.ALL["3d_humanoid_9_full"], 4), ([-1] + list(range(14)), 3)]     # 2 limbs, <= 12 limbs, 15 limbs (chain15)


def _packed_batch():
    graphs = [G.build_graph(par, device="cuda") for par, _ in PACKED]
    tb = make_packed_tables([(gr, B) for gr, (_, B) in zip(graphs, PACKED)], "cuda")
    batches = [synth.make_batch(B, len(par), seed=21 + i) for i, (par, B) in enumerate(PACKED)]
    obs = torch.cat([bt["obs"].view(-1, 41) for bt in batches]).cuda().contiguous()
    act = torch.cat([bt["action"].view(-1, 3) for bt in batches]).cuda().contiguous()
    return graphs, batches, tb, obs, act


@pytest.mark.parametrize("kind", ["critic", "actor"])
def test_packed_ragged_tables_through_backward_raw(mods, kind):
    actor, critic, pa, pc = mods
    graphs, batches, tb, obs, act = _packed_batch()
    assert tb.nmax == 15 and {p[4] for p in tb.parts} == {2, 9, 15}
    mod, nb, od = (critic, 2, 1) if kind == "critic" else (actor, 1, 3)
    out, stash = mod.forward_raw(tb, obs, act if kind == "critic" else None, keep=True, nb=nb)
    dout = torch.randn(nb, tb.T, od, generator=torch.Generator().manual_seed(9)).cuda()
    dobs = torch.full((nb, tb.T, 41), float("nan"), device="cuda")
    mod.backward_raw(tb, stash, dout, nb, None, False, dobs=dobs)
    torch.cuda.synchronize()
    assert torch.isfinite(dobs).all()
    for (t0, t1, _, _, n), gr, bt in zip(tb.parts, graphs, batches):
        B = bt["obs"].shape[0]
        g64 = _g64(gr)
        for z in range(nb):
            if kind == "critic":
                p64 = _p64({k: v for k, v in pc.items() if k.startswith(f"critic{z + 1}.")})
                d = dout[z, t0:t1].double().view(B, n)
                (ds,) = _oracle_input_grads(lambda s_: (O.critic_forward(p64, s_, bt["action"].cuda().double(), g64, which=(z + 1,)) * d).sum(),
                                            bt["obs"].cuda())
            else:
                p64 = _p64(pa)
                d = dout[z, t0:t1].double().reshape(B, n * 3)
                (ds,) = _oracle_input_grads(lambda s_: (O.actor_forward(p64, s_, g64) * d).sum(), bt["obs"].cuda())
            assert parity.rel_err(dobs[z, t0:t1].reshape(B, n * 41), ds) < parity.RTOL, (kind, n, z)


# ---------------------------------------------------------------------------------------------------------------- nothing else moves
@pytest.mark.parametrize("kind", ["critic", "actor"])
def test_dobs_changes_nothing_else_and_costs_one_launch(mods, kind):
    actor, critic, _, _ = mods
    lib = _lib.lib
    par = M.ALL["3d_humanoid_9_full"]
    g = G.build_graph(par, device="cuda")
    b = gpu_util.to_cuda(synth.make_batch(64, len(par), seed=4))
    mod, nb, od = (critic, 2, 1) if kind == "critic" else (actor, 1, 3)
    mod.change_morphology(g)
    tb = mod._tables(64)
    obs = b["obs"].view(-1, 41).contiguous()
    act = b["action"].view(-1, 3).contiguous() if kind == "critic" else None
    dout = torch.randn(nb, tb.T, od, generator=torch.Generator().manual_seed(3)).cuda()
    prev = lib.sgrl_deterministic(1)
    try:
        def run(how):
            _, stash = mod.forward_raw(tb, obs, act, keep=True, nb=nb)
            grads = torch.zeros(mod._nb * mod._live, device="cuda")
            ws = torch.empty(mod.ws_floats(tb.T, nb), device="cuda")
            dact = torch.empty(nb, tb.T, 3, device="cuda") if kind == "critic" else None
            dobs = torch.empty(nb, tb.T, 41, device="cuda") if how == "dobs" else None
            k = mod._call(tb, nb, 1, stash, grads=grads, ws=ws, split=mod._split_for(tb.T, False))
            torch.cuda.synchronize()
            n0 = lib.sgrl_launch_count()
            if how == "legacy":      # the existing entry point
                _lib.check(lib.sgrl_set_backward(C.byref(k), _lib.ptr(dout), tb.T * od, 1, _lib.ptr(dact), tb.T * 3, _lib.stream()))
            else:
                _lib.check(lib.sgrl_set_backward_dobs(C.byref(k), _lib.ptr(dout), tb.T * od, 1, _lib.ptr(dact), tb.T * 3,
                                                      _lib.ptr(dobs), tb.T * 41, _lib.stream()))
            launches = lib.sgrl_launch_count() - n0
            torch.cuda.synchronize()
            return grads, dact, dobs, launches
        g_leg, a_leg, _, n_leg = run("legacy")
        g_none, a_none, _, n_none = run("none")
        g_1, a_1, o_1, n_1 = run("dobs")
        g_2, a_2, o_2, n_2 = run("dobs")
    finally:
        lib.sgrl_deterministic(prev)
    assert n_none == n_leg and n_1 == n_leg + 1 and n_2 == n_1
    assert torch.equal(g_leg, g_none) and torch.equal(g_none, g_1) and torch.equal(g_1, g_2)
    if kind == "critic":
        assert torch.equal(a_leg, a_none) and torch.equal(a_none, a_1) and torch.equal(a_1, a_2)
    assert torch.isfinite(o_1).all() and torch.equal(o_1, o_2)


# ---------------------------------------------------------------------------------------------------------------- torch semantics
def test_state_gradient_accumulates_like_torch(mods, gold):
    _, critic, _, _ = mods
    g, b = _case(gold, "3d_hopper_3_shin", 4)
    critic.change_morphology(g)
    s = b["obs"].clone().requires_grad_(True)
    critic.Q1(s, b["action"]).sum().backward()
    g1 = s.grad.clone()
    critic.Q1(s, b["action"]).sum().backward()
    assert parity.rel_err(s.grad, 2 * g1) < 1e-5


def test_state_gradient_with_frozen_parameters(mods, gold):
    actor, critic, pa, pc = mods
    g, b = _case(gold, "3d_walker_7_full", 5)
    critic.change_morphology(g); actor.change_morphology(g)
    flags = {p: p.requires_grad for m in (actor, critic) for p in m.parameters()}
    actor.zero_grad(set_to_none=True); critic.zero_grad(set_to_none=True)
    try:
        for p in flags:
            p.requires_grad_(False)
        s = b["obs"].clone().requires_grad_(True)
        q = critic.Q1(s, b["action"])
        assert q.grad_fn is not None
        q.sum().backward()
        assert all(p.grad is None for p in critic.parameters())
        pc64, g64 = _p64(pc), _g64(g)
        (ds,) = _oracle_input_grads(lambda s_: O.critic_forward(pc64, s_, b["action"].double(), g64, which=(1,)).sum(), b["obs"])
        assert parity.rel_err(s.grad, ds) < parity.RTOL
        s2 = b["obs"].clone().requires_grad_(True)
        actor(s2).sum().backward()
        pa64 = _p64(pa)
        (ds2,) = _oracle_input_grads(lambda s_: O.actor_forward(pa64, s_, g64).sum(), b["obs"])
        assert parity.rel_err(s2.grad, ds2) < parity.RTOL
    finally:
        for p, f in flags.items():
            p.requires_grad_(f)


def test_twin_critic_dobs_stride_too_small_is_an_error(mods, gold):
    _, critic, _, _ = mods
    g, b = _case(gold, "3d_hopper_3_shin", 4)
    critic.change_morphology(g)
    tb = critic._tables(4)
    _, stash = critic.forward_raw(tb, b["obs"].view(-1, 41).contiguous(), b["action"].view(-1, 3).contiguous(), keep=True, nb=2)
    ws = torch.empty(critic.ws_floats(tb.T, 2), device="cuda")
    dout = torch.ones(2, tb.T, 1, device="cuda")
    dobs = torch.empty(2, tb.T, 41, device="cuda")
    k = critic._call(tb, 2, 1, stash, ws=ws)
    n0 = _lib.lib.sgrl_launch_count()
    rc = _lib.lib.sgrl_set_backward_dobs(C.byref(k), _lib.ptr(dout), tb.T, 0, None, 0, _lib.ptr(dobs), 41 * tb.T - 1, _lib.stream())
    assert rc != 0 and b"dobs_stride" in _lib.lib.sgrl_last_error()
    assert _lib.lib.sgrl_launch_count() == n0      # refused before anything was launched
    with pytest.raises(ValueError):
        critic.backward_raw(tb, stash, dout, 2, None, False, ws=ws, dobs=dobs[:1])
