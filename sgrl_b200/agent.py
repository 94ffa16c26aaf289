"""TD3 agent over the SET modules — drop-in for the reference ``agent.Agent`` with
``actor_type == critic_type == 'set'`` (src/agent.py:20-217): same constructor argument,
``update(data_batch, it)``, ``select_action``, ``change_morphology``, ``models2train/eval``,
``try_update_target_network`` and attributes; it is an ``nn.Module`` whose ``state_dict()``
has the reference's 818 keys (src/common/agents.py:7-11, src/common/trainer.py:256-259).

``update`` does not go through autograd: it drives the forward/backward kernels on the flat
arenas directly and finishes with the fused clip+Adam pass and (every ``policy_freq``-th
call) the Polyak pass.  Under ``torch.distributed`` (one process per GPU, NCCL) the flat
gradient arena is all-reduced once per optimizer step, so every rank applies the identical
update (data parallel over replay samples / morphologies, SURVEY.md §8e).
"""
from __future__ import annotations

import ctypes as C
import os
import warnings
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from ._lib import TD3_HPARAMS, check, lib, ptr, stream
from .modules import SECritic, SEPolicy, SetNetModule


def hparam_table(seeds: List[Dict[str, float]]) -> np.ndarray:
    """The rows of the per-seed TD3 table (SgrlTd3Hparams, include/sgrl_b200.h) for seeds[k] = {actor_lr, critic_lr, discount,
    policy_noise, noise_clip, grad_clipping_value, target_smoothing_tau, reward_scale}.  The fp32 fields are rounded exactly
    as the by-value float arguments were, and one_minus_tau = (float)(1.0 - (double)tau) as sgrl_polyak forms it."""
    rows = np.zeros(len(seeds), dtype=TD3_HPARAMS)
    for field, key in (("actor_lr", "actor_lr"), ("critic_lr", "critic_lr"), ("discount", "discount"), ("reward_scale", "reward_scale"),
                       ("policy_noise", "policy_noise"), ("noise_clip", "noise_clip"), ("tau", "target_smoothing_tau"),
                       ("max_norm", "grad_clipping_value")):
        rows[field] = [float(h[key]) for h in seeds]
    rows["one_minus_tau"] = 1.0 - rows["tau"].astype(np.float64)
    return rows


class FusedAdam:
    """torch.optim.Adam(lr, betas=(0.9,0.999), eps=1e-8) + clip_grad_norm_ over a module's flat
    live arena in one kernel pass (src/agent.py:104-105,152-156,172-176).  groups = K > 1: the module's nets are K independent
    optimizers' parameters (seed-batched agents), net z clipped by the norm over the nets z' with z' % K == z % K."""

    def __init__(self, module: SetNetModule, lr: float, betas=(0.9, 0.999), eps: float = 1e-8, groups: int = 1):
        self.module = module
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.groups = int(groups)
        self._alloc()

    def _alloc(self):
        live = self.module.live_arena
        self.exp_avg = torch.zeros_like(live)
        self.exp_avg_sq = torch.zeros_like(live)
        self.step_count = torch.zeros(1, dtype=torch.int32, device=live.device)
        self.sumsq = torch.zeros(self.module._nb if self.groups > 1 else 1, dtype=torch.float32, device=live.device)   # per net
        self._arena_ptr = live.data_ptr()

    def _sync_device(self):
        if self.module.live_arena.data_ptr() != self._arena_ptr:      # module was moved / re-flattened
            old = (self.exp_avg, self.exp_avg_sq, self.step_count)
            self._alloc()
            self.exp_avg.copy_(old[0]); self.exp_avg_sq.copy_(old[1]); self.step_count.copy_(old[2])

    def zero_grad(self, set_to_none: bool = False):
        self._sync_device()
        self.module.grad_arena().zero_()

    def step(self, max_norm: float = 0.0, world_size: int = 1, keep_split: Optional[bool] = None,
             hparams: Optional[torch.Tensor] = None):
        """Clip (if max_norm > 0) and apply one Adam step from module.grad_arena().  keep_split: also rewrite the tf32
        hi/lo split of the parameters (None: if it is fresh now).  A caller that captures this call into a CUDA graph
        passes the decision explicitly and invalidates the split itself when it is False (Agent._run_update).
        hparams: the device table of per-seed TD3 scalars (one SgrlTd3Hparams row per group, Agent._sync_hparams).  Group g's
        learning rate (the actor or critic one, after the module's kind) and clip threshold are then read from row g when the
        kernel runs, in place of self.lr and max_norm, and the gradient norms are always computed."""
        self._sync_device()
        m = self.module
        g, p = m.grad_arena(), m.live_arena
        nets, st = self.sumsq.numel(), stream()
        n_net = p.numel() // nets
        if hparams is not None and hparams.numel() != self.groups * TD3_HPARAMS.itemsize:
            raise ValueError(f"hparams holds {hparams.numel() // TD3_HPARAMS.itemsize} rows for {self.groups} optimizer groups")
        self.sumsq.zero_()
        if max_norm > 0 or hparams is not None:
            check(lib.sgrl_sumsq_nets(ptr(g), n_net, nets, ptr(self.sumsq), st), "sgrl_sumsq_nets")
        check(lib.sgrl_bump_step(ptr(self.step_count), st), "sgrl_bump_step")
        fresh = m.split_is_fresh() if keep_split is None else (keep_split and m._split is not None)
        if not fresh:
            m.invalidate_split()
        hi, lo = (m._split[0], m._split[1]) if fresh else (None, None)     # keep a valid tf32 split valid (else it is rebuilt lazily)
        if hparams is not None:
            check(lib.sgrl_adam_clip_groups_hp(ptr(p), ptr(g), ptr(self.exp_avg), ptr(self.exp_avg_sq), n_net, nets, self.groups,
                                               ptr(self.sumsq), ptr(self.step_count), ptr(hparams), m._kind, self.betas[0], self.betas[1],
                                               self.eps, 1.0 / world_size, ptr(hi), ptr(lo), st), "sgrl_adam_clip_groups_hp")
            return
        check(lib.sgrl_adam_clip_groups(ptr(p), ptr(g), ptr(self.exp_avg), ptr(self.exp_avg_sq), n_net, nets, self.groups, ptr(self.sumsq),
                                        ptr(self.step_count), self.lr, self.betas[0], self.betas[1], self.eps, float(max_norm), 1.0 / world_size,
                                        ptr(hi), ptr(lo), st), "sgrl_adam_clip_groups")

    def state_dict(self):
        return {"step": self.step_count.clone(), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(),
                "lr": self.lr, "betas": self.betas, "eps": self.eps}

    def load_state_dict(self, sd):
        self._sync_device()
        self.step_count.copy_(sd["step"]); self.exp_avg.copy_(sd["exp_avg"]); self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.lr, self.betas, self.eps = sd["lr"], tuple(sd["betas"]), sd["eps"]


def soft_update_network(source: SetNetModule, target: SetNetModule, tau: float, keep_split: Optional[bool] = None,
                        hparams: Optional[torch.Tensor] = None):
    """theta_t <- tau*theta + (1-tau)*theta_t over ALL parameters incl. the dead ones
    (src/common/functional.py:7-10) as one pass over the flat arenas.  keep_split: see FusedAdam.step.
    hparams: the device table of per-seed TD3 scalars (K rows); net z of the modules, live or dead, then takes seed z % K's
    tau from it when the kernel runs, and `tau` is not used."""
    s, t = source.full_arena, target.full_arena
    if s.device.type != "cuda":
        raise RuntimeError("sgrl_b200.soft_update_network needs the modules on a CUDA device (no CPU fallback)")
    fresh = target.split_is_fresh() if keep_split is None else (keep_split and target._split is not None)
    if not fresh:
        target.invalidate_split()
    hi, lo = (target._split[0], target._split[1]) if fresh else (None, None)
    if hparams is not None:
        check(lib.sgrl_polyak_hp(ptr(t), ptr(s), target._nb, target._live, target._dead, ptr(hparams), hparams.numel() // TD3_HPARAMS.itemsize,
                                 ptr(hi), ptr(lo), stream()), "sgrl_polyak_hp")
        return
    check(lib.sgrl_polyak(ptr(t), ptr(s), s.numel(), float(tau), ptr(hi), ptr(lo), target.live_arena.numel(), stream()), "sgrl_polyak")


class _UpdatePlan:
    """Static device state of Agent.update for one (morphology tables, batch size): input staging buffers, activation
    stashes, backward workspace, small result buffers, the three forward streams and the two captured graphs.
    With K = agent.n_seeds seeds every input and result holds K blocks, seed k's at k*T tokens / k*G graphs; the actor
    modules run K nets, the critics 2K = [critic1 of every seed | critic2 of every seed]."""

    def __init__(self, agent: "Agent", tb):
        dev = agent.actor.full_arena.device
        K = agent.n_seeds
        T, G = tb.T, tb.G
        f = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
        self.tb, self.agent = tb, agent
        # (token0, token1, graph0, graph1, limbs) of every (seed, morphology), seed-major: where load() puts each batch
        self.spans = [(k * T + t0, k * T + t1, k * G + g0, k * G + g1, n) for k in range(K) for (t0, t1, g0, g1, n) in tb.parts]
        # inputs as packed tokens: (T,41) observations / (T,3) actions are exactly the reference's (B, N*41) / (B, N*3) rows.
        # One contiguous block [obs | next_obs | action | reward | done] so that a host batch arrives as ONE H2D copy out of a
        # pinned, double-buffered staging block (the reference issues five pageable copies, src/agent.py:119-125)
        sizes = (K * T * 41, K * T * 41, K * T * 3, K * G, K * G)
        self.inbuf = f(sum(sizes))
        self.obs, self.nobs, self.act, self.rew, self.done = (v.view(-1, w) if w else v for v, w in
                                                              zip(torch.split(self.inbuf, sizes), (41, 41, 3, 0, 0)))
        self.h_in = [torch.empty(sum(sizes), dtype=torch.float32, pin_memory=True) for _ in range(2)]
        self.h_np = [tuple(x.numpy() for x in torch.split(h, sizes)) for h in self.h_in]
        self.h_ev = [torch.cuda.Event(), torch.cuda.Event()]
        self.h_turn = 0
        self.noise = f(K * T, 3)
        # target-policy noise drawn inside the smoothing kernel (Philox keyed by seed, counter = draw): graph-replay safe
        self.draw = torch.zeros(1, dtype=torch.int32, device=dev)
        self.seed = (torch.initial_seed() + 0x9E3779B97F4A7C15 * (len(agent._plans) + 1)) & 0xFFFFFFFFFFFFFFFF
        self.rstats = torch.zeros(K, 2, dtype=torch.float64, device=dev)  # per seed {sum, sum of squares} of the scaled rewards
        self.a_t, self.next_action, self.pi = f(K, T, 3), f(K * T, 3), f(K, T, 3)
        self.tq, self.q, self.q1 = f(2 * K, T, 1), f(2 * K, T, 1), f(K, T, 1)
        self.dq, self.dq1, self.dact = f(2 * K, T, 1), f(K, T, 1), f(K, T, 3)
        self.target = f(K * T)
        self.scal = torch.zeros(2 * K, dtype=torch.float32, device=dev)      # critic losses of the seeds, then their actor losses
        ac, cr = agent.actor, agent.critic
        self.stash_at = f(ac.stash_floats(T, False, K))
        self.stash_ct = f(cr.stash_floats(T, False, 2 * K))
        self.stash_c = f(cr.stash_floats(T, True, 2 * K))
        self.stash_a = f(ac.stash_floats(T, True, K))
        self.ws = f(max(cr.ws_floats(T, 2 * K), ac.ws_floats(T, K)))
        self.s1, self.s2, self.s3, self.s_cap = agent._streams(dev)
        self.ev_start, self.ev_a, self.ev_b, self.ev_c = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        # the fused Adam / Polyak passes of this plan also rewrite the tf32 split (decided once per plan: the captured graphs
        # bake the pointers in).  Plans too small for the tcgen05 path leave the split stale; _run_update then marks it so.
        self.keep_split = all(m.use_tc and T >= m.SPLIT_MIN_TOKENS for m in (agent.actor, agent.critic, agent.actor_target, agent.critic_target))
        self.graphs = {}
        self.graph_launches = {}      # (actor_step, rng) [+ (True,) with the per-morphology statistics] -> kernels of this library inside the captured graph
        self.eager_runs = {}
        self.i_dev = None             # row numbers of a packed buffer gather (stage_indices), allocated on first use
        self.part_stats = None        # (K,P,4) fp64 per-morphology statistics (sgrl_td3_part_stats), allocated on first use

    def alloc_part_stats(self):
        """The result buffer and the fork / join events of the per-morphology statistics; outside any capture, before the
        first step that computes them."""
        if self.part_stats is None:
            K, P = self.agent.n_seeds, len(self.tb.parts)
            self.part_stats = torch.full((K, P, 4), float("nan"), dtype=torch.float64, device=self.inbuf.device)
            self.ev_ps_fork, self.ev_ps_join = torch.cuda.Event(), torch.cuda.Event()

    def load(self, batches, noises):
        """Stage the replay batch of every morphology of the plan (host numpy / CPU or device tensors) into the static
        input buffers.  batches[i]: dict obs (B_i, 41 N_i), action (B_i, 3 N_i), next_obs, reward (B_i,1), done (B_i,1);
        seed-major when the agent has several seeds (self.spans).
        Host batches are packed into a pinned staging block and sent as one copy; device batches are copied in place.
        Returns True when noise was injected (False: the smoothing kernel draws it)."""
        parts = self.spans
        if len(batches) != len(parts):
            raise ValueError(f"plan holds {len(parts)} morphologies, got {len(batches)} batches")
        keys = (("obs", 41), ("next_obs", 41), ("action", 3))
        on_host = all(not (torch.is_tensor(b[k]) and b[k].is_cuda) for b in batches for k in ("obs", "next_obs", "action", "reward", "done"))
        if on_host:
            k = self.h_turn
            self.h_turn ^= 1
            self.h_ev[k].synchronize()                    # the copy that last read this staging block has finished
            h_obs, h_nobs, h_act, h_rew, h_done = self.h_np[k]
            dst_of = {"obs": h_obs, "next_obs": h_nobs, "action": h_act}
        for (t0, t1, g0, g1, n), batch in zip(parts, batches):
            B = g1 - g0
            for key, w in keys:
                src = batch[key]
                if tuple(src.shape) != (B, n * w):
                    raise ValueError(f"{key}: expected {(B, n * w)} for this morphology, got {tuple(src.shape)}")
                if on_host:
                    dst_of[key][t0 * w:t1 * w] = (src.numpy() if torch.is_tensor(src) else np.asarray(src)).reshape(-1)
                else:
                    dst = {"obs": self.obs, "next_obs": self.nobs, "action": self.act}[key]
                    dst[t0:t1].view(B, n * w).copy_(_as_tensor(src), non_blocking=True)
            for key in ("reward", "done"):
                src = batch[key]
                if on_host:
                    (h_rew if key == "reward" else h_done)[g0:g1] = (src.numpy() if torch.is_tensor(src) else np.asarray(src)).reshape(-1)
                else:
                    (self.rew if key == "reward" else self.done)[g0:g1].copy_(_as_tensor(src).reshape(B), non_blocking=True)
        if on_host:
            self.inbuf.copy_(self.h_in[k], non_blocking=True)
            self.h_ev[k].record()
        return self.load_noise(noises)

    def load_noise(self, noises):
        """Target-policy noise of every morphology of the plan (or None: drawn in the smoothing kernel).  Returns True when
        noise was injected."""
        if noises is None or all(nz is None for nz in noises):
            return False
        if len(noises) != len(self.spans):
            raise ValueError(f"plan holds {len(self.spans)} batches, got {len(noises)} noise tensors")
        for (t0, t1, g0, g1, n), nz in zip(self.spans, noises):
            if nz is None:
                raise ValueError("target-policy noise must be given for every morphology of the plan or for none")
            self.noise[t0:t1].view(g1 - g0, n * 3).copy_(_as_tensor(nz).reshape(g1 - g0, n * 3), non_blocking=True)
        return True

    def stage_indices(self, indices):
        """Row numbers of a packed buffer gather (indices[i]: the rows drawn for morphology i) -> self.i_dev, as ONE H2D copy
        out of a pinned, double-buffered block (the pattern of load).  Returns per morphology its slice of the host block."""
        if self.i_dev is None:
            G = self.tb.G * self.agent.n_seeds
            self.i_host = [torch.empty(G, dtype=torch.int64, pin_memory=True) for _ in range(2)]
            self.i_np = [h.numpy() for h in self.i_host]
            self.i_ev = [torch.cuda.Event(), torch.cuda.Event()]
            self.i_turn = 0
            self.i_dev = torch.empty(G, dtype=torch.int64, device=self.inbuf.device)
        k = self.i_turn
        self.i_turn ^= 1
        self.i_ev[k].synchronize()                        # the copy that last read this block has finished
        h = self.i_np[k]
        for (_, _, g0, g1, _), idx in zip(self.spans, indices):
            h[g0:g1] = idx
        self.i_dev.copy_(self.i_host[k], non_blocking=True)
        self.i_ev[k].record()
        return [h[g0:g1] for (_, _, g0, g1, _) in self.spans]

    def replay(self, actor_step: bool, rng: bool, per_morphology: bool = False):
        """per_morphology: the step also computes the per-morphology statistics; such steps have graphs of their own, keyed
        (actor_step, rng, True), so the graphs of the steps without them stay as they are, keyed (actor_step, rng)."""
        key = (actor_step, rng, True) if per_morphology else (actor_step, rng)
        g = self.graphs.get(key)
        if g is None:
            # one eager run first (lazy one-time initialisation inside the library: function attributes, side streams,
            # tensor-map cache), then capture the second
            if self.eager_runs.get(key, 0) < 1:
                self.eager_runs[key] = 1
                self.agent._update_impl(self, actor_step, rng, per_morphology)
                return
            try:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                l0 = lib.sgrl_launch_count()
                with torch.cuda.graph(g, stream=self.s_cap):
                    self.agent._update_impl(self, actor_step, rng, per_morphology)
                self.graph_launches[key] = lib.sgrl_launch_count() - l0
            except Exception as ex:   # keep running eagerly (still the CUDA path); say so once
                warnings.warn(f"sgrl_b200: CUDA-graph capture of Agent.update failed ({ex}); running eagerly")
                self.agent.use_graphs = False
                torch.cuda.synchronize()
                self.agent._update_impl(self, actor_step, rng, per_morphology)
                return
            self.graphs[key] = g
            self.agent.graph_replayed_launches -= self.graph_launches[key]   # the capture itself was counted by the library
        g.replay()
        self.agent.graph_replayed_launches += self.graph_launches[key]


class _RolloutPlan:
    """Static state of the actor's rollout forward for one packed table set: pinned host staging for observations and
    actions, their device twins, the activation scratch, and the captured graph.  K = agent.n_seeds actors act at once,
    seed k on the k-th block of T tokens."""

    def __init__(self, agent: "Agent", tb):
        ac = agent.actor
        dev = ac.full_arena.device
        self.tb, self.agent = tb, agent
        K, T = agent.n_seeds, tb.T
        self.spans = [(k * T + t0, k * T + t1, g0, g1, n) for k in range(K) for (t0, t1, g0, g1, n) in tb.parts]
        self.h_obs = torch.zeros(K * T, 41, dtype=torch.float32, pin_memory=True)
        self.h_out = torch.zeros(K * T, 3, dtype=torch.float32, pin_memory=True)
        self.h_obs_np, self.h_out_np = self.h_obs.numpy().reshape(-1), self.h_out.numpy().reshape(-1)
        self.obs = torch.zeros(K * T, 41, dtype=torch.float32, device=dev)
        self.out = torch.zeros(K, T, 3, dtype=torch.float32, device=dev)
        self.stash = torch.empty(ac.stash_floats(T, False, K), dtype=torch.float32, device=dev)
        self.graph, self.graph_launches, self.eager_runs = None, 0, 0

    def _forward(self):
        K = self.agent.n_seeds
        self.agent.actor.forward_raw(self.tb, self.obs, None, keep=False, nb=K, in_nets=K, trusted_split=True, out=self.out, stash=self.stash)

    def run(self, obs_list):
        """obs_list: one array per part of the table set (env, or the (B,41N) batch of a single-morphology plan), seed-major
        when the agent has several seeds.  Returns per part a numpy view (valid until the next run) of its actions."""
        ag, parts = self.agent, self.spans
        if len(obs_list) != len(parts):
            raise ValueError(f"plan holds {len(parts)} parts, got {len(obs_list)} observations")
        for (t0, t1, _, _, n), o in zip(parts, obs_list):
            o = o.detach().cpu().numpy() if torch.is_tensor(o) else np.asarray(o)
            if o.size != (t1 - t0) * 41:
                raise RuntimeError(f"observation of {o.size} floats for a part of {t1 - t0} limbs x 41")
            self.h_obs_np[t0 * 41:t1 * 41] = o.reshape(-1)           # numpy casts float64 observations (ModularEnv) to fp32 here
        self.obs.copy_(self.h_obs, non_blocking=True)
        ag.actor._split_for(self.tb.T, True)                          # refreshes the tf32 split only if the weights changed
        if not ag.use_graphs:
            self._forward()
        elif self.graph is None and self.eager_runs < 1:
            self.eager_runs += 1
            self._forward()
        else:
            if self.graph is None:
                try:
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    l0 = lib.sgrl_launch_count()
                    with torch.cuda.graph(g):
                        self._forward()
                    self.graph_launches = lib.sgrl_launch_count() - l0
                    ag.graph_replayed_launches -= self.graph_launches
                    self.graph = g
                except Exception as ex:
                    warnings.warn(f"sgrl_b200: CUDA-graph capture of the rollout forward failed ({ex}); running eagerly")
                    ag.use_graphs = False
                    torch.cuda.synchronize()
                    self._forward()
            if self.graph is not None:
                self.graph.replay()
                ag.graph_replayed_launches += self.graph_launches
        self.h_out.copy_(self.out.view(-1, 3), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return [self.h_out_np[t0 * 3:t1 * 3] for (t0, t1, _, _, _) in parts]


class Agent(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        if args.actor_type != "set" or args.critic_type != "set":
            raise NotImplementedError("sgrl_b200 implements the SET actor/critic only (actor_type=critic_type='set')")

        def mk_actor():
            return SEPolicy(args.limb_obs_size, args.limb_action_size, args.msg_dim, args.batch_size, args.max_action,
                            args.max_children, args.disable_fold, args.td, args.bu, args)

        def mk_critic():
            return SECritic(args.limb_obs_size, args.limb_action_size, args.msg_dim, args.batch_size,
                            args.max_children, args.disable_fold, args.td, args.bu, args)

        self.actor, self.actor_target = mk_actor(), mk_actor()
        self.critic, self.critic_target = mk_critic(), mk_critic()
        # sync network parameters (agent.py:100-101, tau = 1.0)
        with torch.no_grad():
            self.actor_target.full_arena.copy_(self.actor.full_arena)
            self.critic_target.full_arena.copy_(self.critic.full_arena)
        self.actor_optimizer = FusedAdam(self.actor, lr=args.lr)
        self.critic_optimizer = FusedAdam(self.critic, lr=args.lr)
        self.n_seeds = 1
        self._init_runtime(args)

    def _init_runtime(self, args):
        """Step state shared by Agent and SeedBatchedAgent: counters, switches and the caches of plans and graphs."""
        self.models2eval()
        self.tot_update_count = 0
        self.target_smoothing_tau = args.agent.target_smoothing_tau
        self.reward_scale = args.agent.reward_scale
        self.data_parallel = True    # False: no gradient all-reduce even inside an initialised process group (tests, replicas-only runs)
        self.lazy_stats = False      # True: reward statistics returned as 0-dim tensors (no host sync)
        self.use_graphs = os.environ.get("SGRL_GRAPHS", "1") != "0"   # replay Agent.update as a captured CUDA graph
        # one plan (static buffers + two or three captured graphs) per (morphology tables, batch size).  The reference's
        # training sets hold up to ~30 morphologies (CWHH++): size the cache from SGRL_MAX_PLANS, evict least recently used
        self.max_plans = max(1, int(os.environ.get("SGRL_MAX_PLANS", "32")))
        self._plans: Dict = {}
        self._packed_tables: Dict = {}
        self._plan_sig = None
        self.graph_replayed_launches = 0     # library kernels executed through graph replays (sgrl_launch_count() sees captures only)
        self._rollout_plans: Dict = {}
        self._rollout_tables: Dict = {}
        self._rollout_sig = None
        self._loss = None
        self._hp = None              # device table of the per-seed TD3 scalars (_sync_hparams), and the rows it holds
        self._hp_rows = None

    # ------------------------------------------------------------------ TD3 step
    def _world(self):
        import torch.distributed as dist
        if not self.data_parallel:
            return 1
        return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1

    def _streams(self, dev):
        """The step's streams, shared by every plan of the agent: s1 carries the critical chain (actor-target ->
        twin critic-target, src/agent.py:127-139), s2 the actor forward of the delayed step, s3 the critic forward, and the
        capture stream the loss / backward / optimizer chain."""
        st = getattr(self, "_stream_set", None)
        if st is None or st[0] != dev:
            st = (dev,) + tuple(torch.cuda.Stream(device=dev) for _ in range(4))
            self._stream_set = st
        return st[1:]

    def _allreduce(self, g: torch.Tensor, world: int):
        if world > 1:
            import torch.distributed as dist
            # eager runs only (no-op under capture): the collective's stream waits on an event recorded right after
            # programmatic-launch kernels, the case csrc/net.cuh stream_fence exists for
            if g.is_cuda:
                check(lib.sgrl_stream_fence(stream()))
            dist.all_reduce(g, op=dist.ReduceOp.SUM)

    def _backward_allreduce(self, module, tb, stash, dout, nb, ws, world):
        """loss.backward() + the data-parallel gradient sum (src/agent.py:151, 171): one flat all-reduce of the gradient arena
        after the backward."""
        g = module.grad_arena()
        module.backward_raw(tb, stash, dout, nb, g, False, trusted_split=True, ws=ws)
        self._allreduce(g, world)

    def _seed_hparams(self) -> List[Dict[str, float]]:
        """The per-step TD3 scalars of every seed, read before each update.  An Agent takes them from its attributes, so a
        change made between updates applies to a replayed CUDA graph as it does eagerly."""
        a = self.args
        return [dict(actor_lr=self.actor_optimizer.lr, critic_lr=self.critic_optimizer.lr, discount=a.discount, policy_noise=a.policy_noise,
                     noise_clip=a.noise_clip, grad_clipping_value=a.grad_clipping_value, target_smoothing_tau=self.target_smoothing_tau,
                     reward_scale=self.reward_scale)]

    def _sync_hparams(self, dev) -> torch.Tensor:
        """The device table the step's kernels read the TD3 scalars from (one SgrlTd3Hparams row per seed, allocated once per
        device).  The rows of _seed_hparams() are copied in stream order when they differ from the rows last copied: in steady
        state nothing is copied."""
        rows = hparam_table(self._seed_hparams()).tobytes()
        if self._hp is None or self._hp.device != dev:
            self._hp = torch.zeros(len(rows), dtype=torch.uint8, device=dev)
            self._hp_rows = None
        if rows != self._hp_rows:
            # pageable source: the copy has staged it when copy_ returns, so a later change cannot race the transfer
            self._hp.copy_(torch.frombuffer(bytearray(rows), dtype=torch.uint8), non_blocking=True)
            self._hp_rows = rows
        return self._hp

    def _plan(self, tb) -> "_UpdatePlan":
        key = id(tb)
        plan = self._plans.get(key)
        if plan is None or plan.tb is not tb:
            while len(self._plans) >= self.max_plans:      # least recently used plan goes (one entry, not the whole cache)
                self._plans.pop(next(iter(self._plans)))
            plan = _UpdatePlan(self, tb)
        else:
            self._plans.pop(key)
        self._plans[key] = plan                            # dicts keep insertion order: most recently used last
        return plan

    def update(self, data_batch: Dict, it: int, noise: Optional[torch.Tensor] = None):
        """One TD3 update (src/agent.py:117-183) on the current morphology (change_morphology).  data_batch: obs (B,41N),
        action (B,3N), next_obs, reward (B,1), done (B,1) — torch tensors (any device) or numpy arrays.  `noise` (B,3N)
        optionally injects the target-policy noise (drawn on device otherwise).

        The batch is copied into a static per-(morphology, B) plan (inputs, activation stashes, workspaces), then
        the whole step runs as ONE captured CUDA graph (two graphs per plan: with and without the delayed actor
        step) — three forward chains on parallel streams, weight-gradient GEMMs on side streams (csrc/net.cuh).
        `self.use_graphs = False` runs the same sequence eagerly."""
        B = int(data_batch["obs"].shape[0])
        tb = self.actor._tables(B)
        return self._run_update(tb, [data_batch], it, None if noise is None else [noise])[0]

    def update_packed(self, batches, it: int, noises=None, morph_count: Optional[float] = None, per_morphology: bool = False):
        """One TD3 update on a PACKED batch of several morphologies: batches = [(graph_dict, data_batch), ...].  The loss is
        the mean over morphologies of the reference's per-morphology loss, so the gradient equals the average of the
        gradients of the separate updates the reference performs one after the other (src/trainer.py:245-250) at the same
        parameters; the limb-tokens of all morphologies go through every kernel together (SURVEY.md §8f rank 1).
        morph_count: data-parallel ranks holding different numbers of morphologies pass (total morphologies / world) so the
        all-reduced gradient is the mean over all morphologies (modules.make_packed_tables).
        per_morphology: the loss dict also holds "per_morphology", one dict per morphology in the order of `batches` with the
        keys a per-morphology Agent.update returns (src/agent.py:158-162, 180): that morphology's critic loss, actor loss
        (actor steps), and the mean and unbiased variance of its scaled rewards.  Floats from one device read per call, or
        0-dim fp64 device tensors with `lazy_stats`.  They do not depend on morph_count and are not all-reduced."""
        tb = self._packed_tables_for([(g, int(b["obs"].shape[0])) for g, b in batches], morph_count)
        return self._run_update(tb, [b for _, b in batches], it, noises, per_morphology=per_morphology)[0]

    def _packed_tables_for(self, specs, morph_count):
        """Packed tables of specs = [(graph_dict, batch size), ...], cached per (graphs, batch sizes, morph_count).
        update_packed and update_packed_from_buffers share the cache, so equal shapes share one plan and its graphs."""
        from .modules import make_packed_tables
        key = tuple((id(g.get("relation")), tuple(g["parents"]), B) for g, B in specs) + (morph_count,)
        tb = self._packed_tables.get(key)
        if tb is None:
            while len(self._packed_tables) >= self.max_plans:
                self._packed_tables.pop(next(iter(self._packed_tables)))
            tb = make_packed_tables(specs, self.actor.full_arena.device, morph_count)
            self._packed_tables[key] = tb
        return tb

    def update_packed_from_buffers(self, parts, batch_size: int, it: int, noises=None, morph_count: Optional[float] = None,
                                   sequential: bool = False, allow_duplicate: bool = False, per_morphology: bool = False):
        """``update_packed([(g, buffer.sample(batch_size)) for g, buffer in parts], it, noises, morph_count, per_morphology)`` without
        materialising the batches: parts = [(graph_dict, sgrl_b200.buffer.ReplayBuffer), ...], one device buffer per morphology
        like the reference keeps them (src/main.py:141-155, src/trainer.py:239-253).  The indices are drawn buffer by buffer in
        list order, exactly as the reference draws them (equal seeds give equal batches; a buffer holding fewer than batch_size
        rows gives a smaller batch), sent as ONE H2D copy, and ONE gather launch writes the rows of all buffers into the static
        inputs of the packed update's plan, which update_packed shares.  Per step: one copy and one launch outside the graph."""
        from .buffer import check_packed_buffers, gather_packed_into
        dev = self.actor.full_arena.device
        buffers = [buf for _, buf in parts]
        check_packed_buffers(buffers, dev)
        for i, (g, buf) in enumerate(parts):
            n = len(g["parents"])
            if buf.obs_dim != 41 * n or buf.action_dim != 3 * n:
                raise ValueError(f"buffer {i} rows ({buf.obs_dim} obs, {buf.action_dim} action floats) do not match its "
                                 f"morphology ({n} limbs)")
            if buf.max_sample_size == 0:
                raise ValueError(f"buffer {i} is empty")
        idx = [buf.draw_indices(batch_size, sequential, allow_duplicate) for buf in buffers]
        tb = self._packed_tables_for([(g, len(ix)) for (g, _), ix in zip(parts, idx)], morph_count)

        def load(plan):
            rows = plan.stage_indices(idx)
            gather_packed_into(buffers, rows, plan.obs, plan.act, plan.nobs, plan.rew, plan.done, idx_dev=plan.i_dev)
            return plan.load_noise(noises)

        return self._run_update(tb, None, it, None, loader=load, per_morphology=per_morphology)[0]

    def update_from_buffer(self, buffer, batch_size: int, it: int, noise: Optional[torch.Tensor] = None,
                           sequential: bool = False, allow_duplicate: bool = False):
        """``update(buffer.sample(batch_size), it)`` (src/trainer.py:289-293) without materialising the batch: the indices are
        drawn like the reference draws them (buffer.py:87-101), and ONE gather kernel writes the sampled rows of the
        device-resident ``sgrl_b200.buffer.ReplayBuffer`` straight into the static input buffers of the update's CUDA
        graph (SURVEY.md §8f rank 2).  Per step the host sends batch_size int64 indices and nothing else."""
        idx = buffer.draw_indices(batch_size, sequential, allow_duplicate)
        B, n = len(idx), self.actor.num_limbs
        if buffer.obs_dim != 41 * n or buffer.action_dim != 3 * n:
            raise ValueError(f"buffer rows ({buffer.obs_dim} obs, {buffer.action_dim} action floats) do not match the current "
                             f"morphology ({n} limbs)")
        tb = self.actor._tables(B)

        def load(plan):
            buffer.gather_into(idx, plan.obs, plan.act, plan.nobs, plan.rew, plan.done)
            if noise is None:
                return False                                                          # drawn in the smoothing kernel (agent.py:128)
            plan.noise.view(B, n * 3).copy_(torch.as_tensor(noise, dtype=torch.float32).reshape(B, n * 3), non_blocking=True)
            return True

        return self._run_update(tb, None, it, None, loader=load)[0]

    def _run_update(self, tb, batches, it: int, noises, loader=None, per_morphology: bool = False):
        """The step of every seed; returns one loss dict per seed (per_morphology: see update_packed)."""
        a = self.args
        dev = self.actor.full_arena.device
        if dev.type != "cuda":
            raise RuntimeError("sgrl_b200.Agent.update needs the modules on a CUDA device (no CPU fallback)")
        mods = (self.actor, self.actor_target, self.critic, self.critic_target)
        # the plans (and their captured graphs) hold raw pointers: drop them when a module was moved / re-flattened or
        # its GEMM path changed.  Parameters edited from Python only stale the tf32 split: in-place torch writes and
        # load_state_dict are detected (SetNetModule._write_stamp), writes through p.data need module.invalidate_split()
        for m in mods:
            m._split_for(tb.T, True)
        hp = self._sync_hparams(dev)
        sig = tuple((m._arena.data_ptr(), int(m.use_tc), 0 if m._split is None else m._split.data_ptr()) for m in mods) + (hp.data_ptr(),)
        if sig != self._plan_sig:
            self._plans.clear()
            self._plan_sig = sig
        plan = self._plan(tb)
        if per_morphology:
            plan.alloc_part_stats()
        injected = loader(plan) if loader is not None else plan.load(batches, noises)
        actor_step = it % a.policy_freq == 0
        if self.use_graphs:
            plan.replay(actor_step, not injected, per_morphology)
        else:
            self._update_impl(plan, actor_step, not injected, per_morphology)
        if plan.keep_split:       # the step's fused Adam / Polyak kernels rewrote hi/lo from the new parameters
            self.critic.mark_split_fresh()
            if actor_step:
                for m in (self.actor, self.critic_target, self.actor_target):
                    m.mark_split_fresh()
        else:
            for m in (self.critic,) + ((self.actor, self.critic_target, self.actor_target) if actor_step else ()):
                m.invalidate_split()
        K, P = self.n_seeds, len(tb.parts)
        scal = plan.scal.clone()
        rewards = [[b["reward"] for b in batches[k * P:(k + 1) * P]] for k in range(K)] if batches is not None else [[plan.rew]] * K
        loss_dicts = []
        for k, stats in enumerate(self._reward_stats(rewards, plan)):
            loss_dict = {"loss/critic_loss": scal[k]}
            loss_dict.update(stats)
            if actor_step:
                loss_dict["loss/actor_loss"] = scal[K + k]
            loss_dicts.append(loss_dict)
        if per_morphology:
            # plan.part_stats[k, i] = {critic loss, actor loss, reward mean, reward variance}: one read for every seed and part
            ps = plan.part_stats.clone() if self.lazy_stats else plan.part_stats.cpu().tolist()
            cols = ((0, "loss/critic_loss"), (2, "misc/train_reward_mean"), (3, "misc/train_reward_var")) + (((1, "loss/actor_loss"),) if actor_step else ())
            for k, loss_dict in enumerate(loss_dicts):
                loss_dict["per_morphology"] = [{key: ps[k][i][j] for j, key in cols} for i in range(P)]
        self.tot_update_count += 1
        self._last_target = plan.target
        return loss_dicts

    def _update_impl(self, p: "_UpdatePlan", actor_step: bool, rng: bool = False, per_morphology: bool = False):
        """Enqueue one update on the current stream (+ p.s1, p.s2 and the library's side streams).  Capture-safe:
        no allocation, no host synchronisation.  The per-seed TD3 scalars are read from the table self._hp when the kernels
        run (_run_update fills it); only max_action and policy_freq are baked in.  per_morphology: one more launch,
        sgrl_td3_part_stats into p.part_stats, on p.s3 (_part_stats)."""
        a = self.args
        hp = self._hp
        tb, T, st = p.tb, p.tb.T, stream()
        K = self.n_seeds          # actor modules: K nets; critics: 2K, net z reading seed z % K's batch
        world = self._world()
        main = torch.cuda.current_stream()
        p.scal.zero_()
        p.ev_start.record(main)
        # ---- chain A (stream s1): y = r + (1-d) * gamma * min_i Q_i'(s', clip(pi'(s') + clip(eps)))        agent.py:127-139
        with torch.cuda.stream(p.s1):
            p.s1.wait_event(p.ev_start)
            self.actor_target.forward_raw(tb, p.nobs, None, keep=False, nb=K, in_nets=K, trusted_split=True, out=p.a_t, stash=p.stash_at)
            if rng:       # eps ~ N(0, policy_noise^2) drawn in the kernel (each seed its own draws); p.noise receives it (tests, logging)
                check(lib.sgrl_bump_step(ptr(p.draw), stream()))
                check(lib.sgrl_td3_smooth_action_rng_hp(ptr(p.a_t), ptr(p.next_action), ptr(p.noise), ptr(hp), T * 3, float(a.max_action),
                                                        K * T * 3, p.seed, ptr(p.draw), stream()))
            else:
                check(lib.sgrl_td3_smooth_action_hp(ptr(p.a_t), ptr(p.noise), ptr(p.next_action), ptr(hp), T * 3, float(a.max_action), K * T * 3,
                                                    stream()))
            self.critic_target.forward_raw(tb, p.nobs, p.next_action, keep=False, nb=2 * K, in_nets=K, trusted_split=True, out=p.tq,
                                           stash=p.stash_ct)
            check(lib.sgrl_stream_fence(stream()))       # eager runs only (no-op under capture): see csrc/net.cuh stream_fence
            p.ev_a.record(p.s1)
        # ---- chain C (stream s2, delayed actor step only): pi(s) — independent of the critic step           agent.py:167
        if actor_step:
            with torch.cuda.stream(p.s2):
                p.s2.wait_event(p.ev_start)
                self.actor.forward_raw(tb, p.obs, None, keep=True, nb=K, in_nets=K, trusted_split=True, out=p.pi, stash=p.stash_a)
                check(lib.sgrl_stream_fence(stream()))
                p.ev_c.record(p.s2)
        # ---- chain B (stream s3, then main): critic step                                                    agent.py:142-156
        with torch.cuda.stream(p.s3):
            p.s3.wait_event(p.ev_start)
            self.critic.forward_raw(tb, p.obs, p.act, keep=True, nb=2 * K, in_nets=K, trusted_split=True, out=p.q, stash=p.stash_c)
            check(lib.sgrl_stream_fence(stream()))
            p.ev_b.record(p.s3)
        main.wait_event(p.ev_b)
        main.wait_event(p.ev_a)
        check(lib.sgrl_td3_critic_loss_seeds_hp(ptr(p.q), ptr(p.tq), ptr(p.rew), ptr(p.done), ptr(tb.tok_graph), ptr(tb.tok_weight),
                                                ptr(p.target), ptr(p.dq), ptr(p.scal), ptr(hp), T, ptr(p.rstats), tb.G, K, st))
        if per_morphology and not actor_step:
            self._part_stats(p, None)
        self.critic_optimizer.zero_grad()
        self._backward_allreduce(self.critic, tb, p.stash_c, p.dq, 2 * K, p.ws, world)
        self.critic_optimizer.step(world_size=world, keep_split=p.keep_split, hparams=hp)
        # ---- delayed actor step + Polyak                                                                    agent.py:165-180
        if actor_step:
            main.wait_event(p.ev_c)
            # critic1 of every seed = the first K nets of the critic arena
            self.critic.forward_raw(tb, p.obs, p.pi, keep=True, nb=K, in_nets=K, trusted_split=True, out=p.q1, stash=p.stash_c)
            check(lib.sgrl_td3_actor_loss_seeds(ptr(p.q1), ptr(tb.tok_weight), ptr(p.dq1), ptr(p.scal[K:]), T, K, st))
            if per_morphology:
                self._part_stats(p, p.q1)
            self.critic.backward_raw(tb, p.stash_c, p.dq1, K, None, True, trusted_split=True, ws=p.ws, dact=p.dact)   # only d/d(action)
            self.actor_optimizer.zero_grad()
            self._backward_allreduce(self.actor, tb, p.stash_a, p.dact, K, p.ws, world)
            self.actor_optimizer.step(world_size=world, keep_split=p.keep_split, hparams=hp)
            self.try_update_target_network(keep_split=p.keep_split, hparams=hp)
        if per_morphology:
            main.wait_event(p.ev_ps_join)

    def _part_stats(self, p: "_UpdatePlan", q1):
        """Per-morphology statistics of the step (sgrl_td3_part_stats) off the critical chain: forked from the current stream to
        p.s3, whose critic forward the current stream has already joined, and joined again at the end of the step.  It reads
        p.q, p.target, p.rew and q1 (p.q1 on actor steps, else None), which nothing later in the step writes."""
        main = torch.cuda.current_stream()
        check(lib.sgrl_stream_fence(stream()))       # eager runs only (no-op under capture): see csrc/net.cuh stream_fence
        p.ev_ps_fork.record(main)
        with torch.cuda.stream(p.s3):
            p.s3.wait_event(p.ev_ps_fork)
            tb = p.tb
            check(lib.sgrl_td3_part_stats(ptr(p.q), ptr(p.target), ptr(q1), ptr(p.rew), ptr(tb.part_table), len(tb.parts), tb.T, tb.G,
                                          self.n_seeds, ptr(self._hp), ptr(p.part_stats), stream()), "sgrl_td3_part_stats")
            check(lib.sgrl_stream_fence(stream()))
            p.ev_ps_join.record(p.s3)

    train_step = update   # BASELINE.json calls the TD3 step "train()"; the reference name is update (agent.py:117)

    def _reward_stats(self, rewards_per_seed, plan):
        """agent.py:158-162 returns Python floats (two device syncs in the reference).  When the batch arrived from host
        memory the statistics are computed there and nothing synchronises; otherwise they come from the sum / sum of
        squares the critic-loss kernel accumulated in fp64 (one 16-byte read per seed, one sync for all of them;
        `lazy_stats`: left on the device).  rewards_per_seed[k]: the reward arrays of seed k, scaled by seed k's reward_scale;
        returns one dict per seed."""
        if all(isinstance(r, np.ndarray) or (torch.is_tensor(r) and not r.is_cuda) for rs in rewards_per_seed for r in rs):
            out = []
            for rewards_in, h in zip(rewards_per_seed, self._seed_hparams()):
                s = h["reward_scale"]
                r = torch.cat([torch.as_tensor(x, dtype=torch.float32).reshape(-1) for x in rewards_in]) * s
                out.append({"misc/train_reward_mean": r.mean().item(), "misc/train_reward_var": r.var().item() if r.numel() > 1 else float("nan")})
            return out
        n = plan.tb.G
        sts = plan.rstats.clone() if self.lazy_stats else plan.rstats.cpu()
        out = []
        for st in sts:
            mean = st[0] / n
            var = (st[1] - st[0] * st[0] / n) / (n - 1) if n > 1 else st[0] * float("nan")
            if self.lazy_stats:
                out.append({"misc/train_reward_mean": mean, "misc/train_reward_var": var})
            else:
                out.append({"misc/train_reward_mean": float(mean), "misc/train_reward_var": float(var)})
        return out

    def try_update_target_network(self, keep_split: Optional[bool] = None, hparams: Optional[torch.Tensor] = None):
        """Polyak update of both target networks with target_smoothing_tau, or (hparams: the device table of _sync_hparams)
        with each seed's tau read when the kernel runs."""
        soft_update_network(self.critic, self.critic_target, self.target_smoothing_tau, keep_split, hparams)
        soft_update_network(self.actor, self.actor_target, self.target_smoothing_tau, keep_split, hparams)

    # ------------------------------------------------------------------ acting
    def _rollout_plan(self, tb) -> "_RolloutPlan":
        sig = (self.actor._arena.data_ptr(), int(self.actor.use_tc))
        if sig != self._rollout_sig:
            self._rollout_plans.clear()
            self._rollout_sig = sig
        plan = self._rollout_plans.get(id(tb))
        if plan is None or plan.tb is not tb:
            while len(self._rollout_plans) >= 64:
                self._rollout_plans.pop(next(iter(self._rollout_plans)))
            plan = _RolloutPlan(self, tb)
            self._rollout_plans[id(tb)] = plan
        return plan

    @torch.no_grad()
    def select_action(self, obs, deterministic=False):
        """src/agent.py:189-198: numpy (41N,) or (B,41N) -> numpy (B,3N).  The forward of one (morphology, B) runs as a
        replayed CUDA graph over pinned staging buffers (one H2D copy, ~70 kernels in one launch, one D2H copy)."""
        if len(obs.shape) == 1:
            obs = obs[None,]
        dev = self.actor.full_arena.device
        if dev.type != "cuda":
            raise RuntimeError("sgrl_b200.Agent.select_action needs the modules on a CUDA device (no CPU fallback)")
        B, n = int(obs.shape[0]), self.actor.num_limbs
        if obs.shape[1] != 41 * n:
            raise RuntimeError(f"shape '[{B}, {n}, -1]' is invalid for input of size {int(np.prod(obs.shape))}")
        if torch.is_tensor(obs) and obs.is_cuda:
            return self.actor(obs).cpu().numpy()
        plan = self._rollout_plan(self.actor._tables(B))
        return plan.run([obs])[0].reshape(B, 3 * n).copy()

    @torch.no_grad()
    def select_actions(self, obs_list, graphs, deterministic=False):
        """Batched rollout front-end (SURVEY.md §8f rank 4).  The reference acts env by env —
        ``change_morphology(graph_i); select_action(obs_i)`` with B=1, src/trainer.py:174-196 and common/trainer.py:93-109 —
        i.e. one ~1 700-op forward and two host<->device round trips per env and step.  Here the observations of ALL envs
        (mixed morphologies) are packed into one ragged batch: obs_list[i] is env i's un-padded (41*N_i,) observation,
        graphs[i] its graph dict; returns [ (1, 3*N_i) numpy action ] in env order.  One pinned H2D copy, one replayed
        CUDA graph of the packed actor forward, one D2H copy.  Exploration noise / zero-padding stay with the caller."""
        if len(obs_list) != len(graphs) or not obs_list:
            raise ValueError("select_actions needs one graph per observation")
        out = self._rollout_plan(self._rollout_tables_for(graphs)).run(obs_list)
        return [o.reshape(1, -1).copy() for o in out]

    def _rollout_tables_for(self, graphs):
        """Packed tables of one env per graph, cached per list of graphs."""
        from .modules import make_packed_tables
        key = tuple((id(g.get("relation")), tuple(g["parents"])) for g in graphs)
        tb = self._rollout_tables.get(key)
        if tb is None:
            while len(self._rollout_tables) >= 64:
                self._rollout_tables.pop(next(iter(self._rollout_tables)))
            tb = make_packed_tables([(g, 1) for g in graphs], self.actor.full_arena.device)
            self._rollout_tables[key] = tb
        return tb

    def change_morphology(self, graph):
        self.actor.change_morphology(graph)
        self.actor_target.change_morphology(graph)
        self.critic.change_morphology(graph)
        self.critic_target.change_morphology(graph)

    def models2eval(self):
        self.actor = self.actor.eval()
        self.actor_target = self.actor_target.eval()
        self.critic = self.critic.eval()
        self.critic_target = self.critic_target.eval()

    def models2train(self):
        self.actor = self.actor.train()
        self.actor_target = self.actor_target.train()
        self.critic = self.critic.train()
        self.critic_target = self.critic_target.train()


def _as_tensor(x):
    return x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x), dtype=torch.float32)


def _to_dev(x, dev):
    if not torch.is_tensor(x):
        x = torch.as_tensor(np.asarray(x), dtype=torch.float32)
        if dev.type == "cuda":
            x = x.pin_memory()
    return x.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
