"""Seed-batched TD3: K independent SET agents trained in one captured update per step.

RL results are reported over seeds (the reference's configs run B = 100 and B = 256).  At those batch sizes one agent's step
is bound by the latency of its kernel chain, not by work, so K agents stepped one after the other cost about K steps.
``SeedBatchedAgent`` stacks the seeds on the executor's net axis instead: the actor modules hold K nets, the critic modules
2K nets ordered [critic1 of seeds 0..K-1 | critic2 of seeds 0..K-1], and every kernel of the step runs once for all seeds,
net z reading seed z % K's batch.  The update sequence is ``Agent._update_impl`` itself (it takes the seed count from
``n_seeds``); clipping and Adam are per seed (one grouped launch each), Polyak and the all-reduce cover the whole arena.

Each seed has its own initial weights (those of ``torch.manual_seed(seed); Agent(args)``), Adam state, target networks,
replay data and target-policy noise, and its own TD3 hyper-parameters (``HPARAM_KEYS``: learning rates, discount, target-policy
noise and its clip, gradient clip, target smoothing tau, reward scale), so one seed-batched agent can run a hyper-parameter
sweep.  The step's kernels read these from a small device table (one row per seed) when they run: ``set_hparams`` between
updates takes effect at the next update without recapturing the step's graphs.  The seeds share the morphology of each step,
``policy_freq``, ``max_action``, Adam's betas and eps, the batch size and the architecture.
"""
from __future__ import annotations

import contextlib
import copy
import ctypes as C
import math
import numbers
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from ._lib import ACTOR, CRITIC, SeedPlane, SgrlError, check, lib, ptr, stream
from .agent import Agent, FusedAdam
from .buffer import MAX_SEEDS
from .modules import SetNetModule


@contextlib.contextmanager
def _rng_kept():
    """Runs its body without changing the caller's CPU / current-CUDA-device random streams."""
    devices = [torch.cuda.current_device()] if torch.cuda.is_available() else []
    with torch.random.fork_rng(devices=devices):
        yield


def _seed_nets(K: int, k: int, per_agent: int):
    """(net z of the seed-batched module, net j of seed k's own module): net j of every seed, then net j + 1."""
    return [(j * K + k, j) for j in range(per_agent)]


def _copy_seed(b: SetNetModule, one: SetNetModule, K: int, k: int, to_batched: bool):
    """Seed k's parameters (live and dead) between a seed-batched module and the seed's own module."""
    L, D = b._live, b._dead
    with torch.no_grad():
        for z, j in _seed_nets(K, k, one._nb):
            for bz, oj in ((b._arena[z * L:(z + 1) * L], one._arena[j * L:(j + 1) * L]),
                           (b._arena[b._nb * L + z * D:b._nb * L + (z + 1) * D], one._arena[one._nb * L + j * D:one._nb * L + (j + 1) * D])):
                (bz if to_batched else oj).copy_(oj if to_batched else bz)


def _copy_seed_adam(b: FusedAdam, one: FusedAdam, K: int, k: int, to_batched: bool):
    """Seed k's Adam moments (live arena only) between a seed-batched optimizer and the seed's own."""
    L = b.module._live
    with torch.no_grad():
        for z, j in _seed_nets(K, k, one.module._nb):
            for bt, ot in ((b.exp_avg, one.exp_avg), (b.exp_avg_sq, one.exp_avg_sq)):
                bz, oj = bt[z * L:(z + 1) * L], ot[j * L:(j + 1) * L]
                (bz if to_batched else oj).copy_(oj if to_batched else bz)


class SeedBatchedAgent(Agent):
    """K = len(seeds) (1..8) independent TD3 agents over the SET modules, stepped together.

    ``update(batches, it)`` performs one TD3 step (src/agent.py:117-183) for every seed as ONE captured CUDA graph and returns
    one loss dict per seed, with the keys ``Agent.update`` returns; ``update_packed_per_seed`` does the same for packed
    multi-morphology batches (``Agent.update_packed`` per seed).  ``agent(k)`` gives seed k as a standalone ``Agent`` (its
    ``state_dict`` has the reference's 818 keys); ``from_agents`` builds a seed-batched agent from existing ones.

    hparams: None (every seed trains with args' values) or K dicts, dict k overriding args for seed k with any of ``lr`` and
    ``HPARAM_KEYS``.  ``get_hparams(k)`` / ``set_hparams(k, **values)`` read and change seed k's values; the step reads them
    before every update.  The Agent attributes that carry these values for a single agent (the optimizers' ``lr``,
    ``args.discount`` and the like, ``target_smoothing_tau``, ``reward_scale``) hold seed 0's initial values and are not read.
    ``exploit({dst: src})`` copies whole seeds onto others in place (population-based training), without recapturing."""

    def __init__(self, args, seeds: Sequence[int], hparams: Optional[Sequence[Dict]] = None):
        seeds = list(seeds)
        _check_count(len(seeds))
        base = args_hparams(args)
        if hparams is None:
            per_seed = [dict(base) for _ in seeds]
        else:
            hparams = list(hparams)
            if len(hparams) != len(seeds):
                raise ValueError(f"hparams: expected one dict per seed ({len(seeds)}), got {len(hparams)}")
            per_seed = [{**base, **check_hparams(h, f"hparams[{k}]")} for k, h in enumerate(hparams)]
        agents = []
        with _rng_kept():
            for sd in seeds:
                torch.manual_seed(sd)
                agents.append(Agent(args))
        self._init_from(agents, per_seed)

    @classmethod
    def from_agents(cls, agents: Sequence[Agent]) -> "SeedBatchedAgent":
        """A seed-batched copy of existing agents: parameters, target networks, Adam moments and step counts, and each agent's
        own hyper-parameters (its optimizers' lr, args' discount, policy noise, noise clip and gradient clip, its
        target_smoothing_tau and reward_scale).  The agents must share policy_freq and max_action and have taken the same
        number of optimizer steps (the seeds share one step counter)."""
        agents = list(agents)
        _check_count(len(agents))
        for key in ("policy_freq", "max_action"):
            values = {getattr(a.args, key) for a in agents}
            if len(values) != 1:
                raise ValueError(f"the agents' {key} differ ({sorted(values)}): every seed of a SeedBatchedAgent shares it")
        for name in ("actor_optimizer", "critic_optimizer"):
            steps = {int(getattr(a, name).step_count.item()) for a in agents}
            if len(steps) != 1:
                raise ValueError(f"the agents' {name} step counts differ ({sorted(steps)}): seed-batched agents step together")
        self = cls.__new__(cls)
        self._init_from(agents, [a._seed_hparams()[0] for a in agents])
        return self

    def _init_from(self, agents: List[Agent], per_seed: List[Dict[str, float]]):
        nn_init = super(Agent, self).__init__          # nn.Module.__init__: the modules are built here, not by Agent.__init__
        nn_init()
        a0 = agents[0]
        args = a0.args
        K = len(agents)
        dev = a0.actor.full_arena.device
        self.args, self.n_seeds = args, K
        with _rng_kept():                               # the arenas are overwritten below: their own init draws nothing visible
            self.actor = SetNetModule(ACTOR, [f"actor_{k}" for k in range(K)], args, max_action=args.max_action, device=dev)
            self.actor_target = SetNetModule(ACTOR, [f"actor_{k}" for k in range(K)], args, max_action=args.max_action, device=dev)
            names = [f"critic{j + 1}_{k}" for j in range(2) for k in range(K)]
            self.critic = SetNetModule(CRITIC, names, args, device=dev)
            self.critic_target = SetNetModule(CRITIC, names, args, device=dev)
        for m in ("actor", "actor_target", "critic", "critic_target"):
            for k, a in enumerate(agents):
                _copy_seed(getattr(self, m), getattr(a, m), K, k, True)
            getattr(self, m).use_tc = getattr(a0, m).use_tc
        self.actor_optimizer = FusedAdam(self.actor, lr=a0.actor_optimizer.lr, betas=a0.actor_optimizer.betas, eps=a0.actor_optimizer.eps,
                                         groups=K)
        self.critic_optimizer = FusedAdam(self.critic, lr=a0.critic_optimizer.lr, betas=a0.critic_optimizer.betas,
                                          eps=a0.critic_optimizer.eps, groups=K)
        for name in ("actor_optimizer", "critic_optimizer"):
            opt = getattr(self, name)
            for k, a in enumerate(agents):
                _copy_seed_adam(opt, getattr(a, name), K, k, True)
            opt.step_count.copy_(getattr(a0, name).step_count)
        self._init_runtime(args)
        self.tot_update_count = a0.tot_update_count
        self.target_smoothing_tau, self.reward_scale = a0.target_smoothing_tau, a0.reward_scale
        self._hparams = [{key: float(h[key]) for key in HPARAM_KEYS} for h in per_seed]
        if hasattr(a0.actor, "graph"):
            self.change_morphology(a0.actor.graph)

    def _check_index(self, k: int):
        if not 0 <= k < self.n_seeds:
            raise ValueError(f"seed index {k} outside 0..{self.n_seeds - 1}")

    def get_hparams(self, k: int) -> Dict[str, float]:
        """Seed k's hyper-parameters, {HPARAM_KEYS key: value} (a copy)."""
        self._check_index(k)
        return dict(self._hparams[k])

    def set_hparams(self, k: int, **values):
        """Changes seed k's hyper-parameters (keywords as in the constructor's hparams dicts).  The next update uses them: the
        step's graphs read them from the device table, which is rewritten in stream order before that update; nothing is
        recaptured.  Raises ValueError, changing nothing, on a key or value the constructor refuses."""
        self._check_index(k)
        self._hparams[k].update(check_hparams(values, f"set_hparams({k})"))

    def _seed_hparams(self) -> List[Dict[str, float]]:
        return self._hparams

    def try_update_target_network(self, keep_split: Optional[bool] = None, hparams=None):
        """Polyak update of every seed's target networks with its own tau."""
        if hparams is None:
            hparams = self._sync_hparams(self.actor.full_arena.device)
        super().try_update_target_network(keep_split, hparams)

    def agent(self, k: int) -> Agent:
        """Seed k as a standalone ``Agent`` (a copy): parameters, target networks, Adam state, update count and hyper-parameters
        (in a copy of args and in the optimizers' lr)."""
        self._check_index(k)
        dev = self.actor.full_arena.device
        h = self._hparams[k]
        with _rng_kept():
            a = Agent(args_with(self.args, h))
        a.to(dev)
        for m in ("actor", "actor_target", "critic", "critic_target"):
            _copy_seed(getattr(self, m), getattr(a, m), self.n_seeds, k, False)
            getattr(a, m).use_tc = getattr(self, m).use_tc
        for name in ("actor_optimizer", "critic_optimizer"):
            mine, one = getattr(self, name), getattr(a, name)
            one._sync_device()
            _copy_seed_adam(mine, one, self.n_seeds, k, False)
            one.step_count.copy_(mine.step_count)
            one.lr, one.betas, one.eps = h["actor_lr" if name == "actor_optimizer" else "critic_lr"], mine.betas, mine.eps
        a.tot_update_count = self.tot_update_count
        a.target_smoothing_tau, a.reward_scale = h["target_smoothing_tau"], h["reward_scale"]
        a.data_parallel, a.lazy_stats, a.use_graphs = self.data_parallel, self.lazy_stats, self.use_graphs
        if hasattr(self.actor, "graph"):
            a.change_morphology(self.actor.graph)
        return a

    # ------------------------------------------------------------------ population-based training
    def exploit(self, pairs: Dict[int, int]):
        """The exploit step of population-based training: for every dst: src of `pairs`, seed dst becomes a bit-for-bit copy of
        seed src's training state: the online actor and twin critics (live and dead parameters), the target networks, both
        optimizers' Adam moments, the tf32 weight splits where allocated, and the hyper-parameters (get_hparams(dst) ==
        get_hparams(src) afterwards).  Explore with set_hparams after it.

        One ``sgrl_seed_copy`` launch on the current stream, in stream order between two updates, and no host synchronisation.
        The copies land in the arenas the plans and their captured graphs already point at, so nothing is reallocated or
        recaptured: the next update replays the graphs it would have replayed anyway, and the changed hyper-parameter rows
        reach the device table before it like any set_hparams change.
        Left as they are: the replay buffers (the caller owns them), the Adam step count and tot_update_count (shared by every
        seed) and each seed's target-policy noise stream (dst keeps drawing its own noise).  The gradient arenas, the
        optimizers' per-net norms and the plans' buffers are not copied: every step overwrites them before reading them.
        Data parallelism: every rank must call exploit with the same mapping (there is no collective), or the replicas
        diverge.

        ValueError, before anything changes, for: `pairs` not a dict, an index that is not an int, an index outside 0..K-1,
        dst == src, a repeated dst, a seed that is both a dst and a src.  An empty dict does nothing.  Off CUDA: SgrlError,
        after these checks, as for every module call without a GPU."""
        mapping = self._check_pairs(pairs)
        if not mapping:
            return
        if self.actor.full_arena.device.type != "cuda":
            raise SgrlError("SeedBatchedAgent.exploit needs the modules on a CUDA device (no CPU fallback)")
        planes = self._seed_planes()
        desc = (SeedPlane * len(planes))(*(SeedPlane(ptr(t), n_net, per, 0) for t, n_net, per in planes))
        n = len(mapping)
        dst = (C.c_int32 * n)(*(d for d, _ in mapping))
        src = (C.c_int32 * n)(*(s for _, s in mapping))
        # The raw writes bump no version counter, so a tf32 split flagged fresh stays flagged fresh.  That is right: a fresh
        # split is an elementwise function of the live parameters, and dst's hi / lo planes are copied with them.  A stale
        # split stays flagged stale and is re-derived before its next use, as it would have been.
        check(lib.sgrl_seed_copy(desc, len(planes), self.n_seeds, dst, src, n, stream()), "sgrl_seed_copy")
        for d, s in mapping:
            self._hparams[d] = dict(self._hparams[s])

    def _check_pairs(self, pairs) -> List[Tuple[int, int]]:
        """exploit's {dst: src} -> [(dst, src)], with the refusals of sgrl_seed_copy as ValueError."""
        if not isinstance(pairs, dict):
            raise ValueError(f"exploit: expected a {{dst: src}} dict of seed indices, got {type(pairs).__name__}")
        out = []
        for d, s in pairs.items():
            for x in (d, s):
                if isinstance(x, bool) or not isinstance(x, numbers.Integral):
                    raise ValueError(f"exploit: seed indices must be ints, got {x!r}")
                self._check_index(int(x))
            if int(d) == int(s):
                raise ValueError(f"exploit: seed {int(d)} would be copied onto itself")
            out.append((int(d), int(s)))
        dsts = [d for d, _ in out]
        if len(set(dsts)) != len(dsts):
            raise ValueError(f"exploit: a dst seed appears twice in {sorted(dsts)}")
        both = set(dsts) & {s for _, s in out}
        if both:
            raise ValueError(f"exploit: seeds {sorted(both)} would both receive and give a copy in one call")
        return out

    def _seed_planes(self) -> List[Tuple[torch.Tensor, int, int]]:
        """Every per-seed state array of the agent, each once, as the planes of sgrl_seed_copy: (tensor, n_net, nets_per_seed),
        net z of the tensor at z * n_net floats, seed k's nets k + j*K for j < nets_per_seed.  Per module its live and its dead
        parameters (the arena is [live nets | dead nets]) and, where allocated, the tf32 split hi and lo of the live ones; per
        optimizer its Adam exp_avg and exp_avg_sq."""
        K = self.n_seeds
        for opt in (self.actor_optimizer, self.critic_optimizer):
            opt._sync_device()              # a moved module: the moments follow it before their pointers are taken
        planes = []
        for m in (self.actor, self.actor_target, self.critic, self.critic_target):
            per, L, D = m._nb // K, m._live, m._dead
            planes.append((m.live_arena, L, per))
            if D:
                planes.append((m.full_arena[m._nb * L:], D, per))
            if m._split is not None:
                planes += [(m._split[0], L, per), (m._split[1], L, per)]
        for opt in (self.actor_optimizer, self.critic_optimizer):
            m = opt.module
            planes += [(opt.exp_avg, m._live, m._nb // K), (opt.exp_avg_sq, m._live, m._nb // K)]
        return planes

    # ------------------------------------------------------------------ TD3 step
    def update(self, batches, it: int, noises=None):
        """One TD3 step of every seed on the current morphology.  batches[k]: seed k's batch as ``Agent.update`` takes it
        (obs (B,41N), action (B,3N), next_obs, reward (B,1), done (B,1)), the same B for every seed.  noises: None (drawn on
        the device, each seed its own draws) or K tensors (B,3N).  Returns K loss dicts; the reward statistics cost one host
        synchronisation for all seeds (none for host batches or with ``lazy_stats``)."""
        self._check_list(batches, "batches")
        if noises is not None:
            self._check_list(noises, "noises")
        sizes = {int(b["obs"].shape[0]) for b in batches}
        if len(sizes) != 1:
            raise ValueError(f"every seed's batch must hold the same number of samples, got {sorted(sizes)}")
        tb = self.actor._tables(sizes.pop())
        return self._run_update(tb, list(batches), it, None if noises is None else list(noises))

    train_step = update

    def update_from_buffers(self, buffers, batch_size: int, it: int, noises=None, sequential: bool = False, allow_duplicate: bool = False):
        """``update([buf.sample(batch_size) for buf in buffers], it, noises)`` without materialising the batches: buffers[k] is
        seed k's device ``sgrl_b200.buffer.ReplayBuffer`` holding transitions of the current morphology.  The indices are drawn
        buffer by buffer with ``buf.draw_indices``, sent as ONE H2D copy, and ONE gather launch writes every seed's rows into
        its block of the step's static inputs."""
        from .buffer import check_packed_buffers, gather_packed_into
        self._check_list(buffers, "buffers")
        if noises is not None:
            self._check_list(noises, "noises")
        check_packed_buffers(buffers, self.actor.full_arena.device)
        n = self.actor.num_limbs
        for k, buf in enumerate(buffers):
            if buf.obs_dim != 41 * n or buf.action_dim != 3 * n:
                raise ValueError(f"buffer {k} rows ({buf.obs_dim} obs, {buf.action_dim} action floats) do not match the current "
                                 f"morphology ({n} limbs)")
            if buf.max_sample_size == 0:
                raise ValueError(f"buffer {k} is empty")
        idx = [buf.draw_indices(batch_size, sequential, allow_duplicate) for buf in buffers]
        sizes = sorted({len(ix) for ix in idx})
        if len(sizes) != 1:
            raise ValueError(f"the buffers gave batches of {sizes} rows: every seed needs the same batch size")
        tb = self.actor._tables(sizes[0])

        def load(plan):
            rows = plan.stage_indices(idx)
            gather_packed_into(buffers, rows, plan.obs, plan.act, plan.nobs, plan.rew, plan.done, idx_dev=plan.i_dev)
            return plan.load_noise(noises)

        return self._run_update(tb, None, it, None, loader=load)

    def update_packed_per_seed(self, batches_per_seed, it: int, noises=None, morph_count: Optional[float] = None,
                               per_morphology: bool = False):
        """``Agent.update_packed`` of every seed in ONE captured step: batches_per_seed[k] is what seed k's own agent would pass
        to update_packed, [(graph_dict, data_batch), ...].  The seeds share the morphologies (the same parents in the same
        order) and the batch size of each; seed 0's graph dicts build the packed tables.  noises: None or K lists of one
        (B_i, 3 N_i) tensor per morphology.  Returns K loss dicts; seed k's loss is the mean over its morphologies, as in
        update_packed.  morph_count and per_morphology: as in ``Agent.update_packed`` (data parallelism; seed k's
        "per_morphology" list holds seed k's own values, its rewards scaled by its own reward_scale)."""
        graphs = self._check_seed_morphologies(batches_per_seed, "batches_per_seed")
        specs = [(g, int(b["obs"].shape[0])) for g, b in batches_per_seed[0]]
        for k, parts in enumerate(batches_per_seed):
            for i, ((_, b), (_, B)) in enumerate(zip(parts, specs)):
                if int(b["obs"].shape[0]) != B:
                    raise ValueError(f"seed {k} morphology {i}: a batch of {int(b['obs'].shape[0])} samples, seed 0's holds {B}: "
                                     f"every seed needs the same batch size per morphology")
        flat_noises = self._seed_noises(noises, len(graphs))
        tb = self._packed_tables_for(specs, morph_count)
        return self._run_update(tb, [b for parts in batches_per_seed for _, b in parts], it, flat_noises, per_morphology=per_morphology)

    def update_packed_from_buffers_per_seed(self, parts_per_seed, batch_size: int, it: int, noises=None,
                                            morph_count: Optional[float] = None, sequential: bool = False, allow_duplicate: bool = False,
                                            per_morphology: bool = False):
        """``update_packed_per_seed([[(g, buf.sample(batch_size)) for g, buf in parts] for parts in parts_per_seed], ...)``
        without materialising the batches: parts_per_seed[k] = [(graph_dict, ReplayBuffer), ...] is seed k's device buffer of
        each morphology.  The indices are drawn with ``buf.draw_indices`` seed after seed, buffer after buffer (the draws of K
        agents calling ``update_packed_from_buffers`` in seed order), sent as ONE H2D copy, and ONE gather launch
        (``gather_seeds_into``) writes every seed's rows into its block of the step's static inputs.  Per step: one copy and
        one library launch outside the graph.  The plan is update_packed_per_seed's, and so is per_morphology."""
        from .buffer import check_seed_buffers, gather_seeds_into
        graphs = self._check_seed_morphologies(parts_per_seed, "parts_per_seed")
        flat_noises = self._seed_noises(noises, len(graphs))
        for k, parts in enumerate(parts_per_seed):
            for i, (g, buf) in enumerate(parts):
                n = len(g["parents"])
                if buf.obs_dim != 41 * n or buf.action_dim != 3 * n:
                    raise ValueError(f"seed {k} buffer {i} rows ({buf.obs_dim} obs, {buf.action_dim} action floats) do not match its "
                                     f"morphology ({n} limbs)")
                if buf.max_sample_size == 0:
                    raise ValueError(f"seed {k} buffer {i} is empty")
        buffers = [[buf for _, buf in parts] for parts in parts_per_seed]
        check_seed_buffers(buffers, self.actor.full_arena.device)
        idx = [[buf.draw_indices(batch_size, sequential, allow_duplicate) for buf in bufs] for bufs in buffers]
        for k in range(1, self.n_seeds):
            for i, (a, b) in enumerate(zip(idx[k], idx[0])):
                if len(a) != len(b):
                    raise ValueError(f"seed {k} buffer {i} gave a batch of {len(a)} rows, seed 0's {len(b)}: every seed needs the "
                                     f"same batch size per morphology")
        tb = self._packed_tables_for([(g, len(ix)) for g, ix in zip(graphs, idx[0])], morph_count)
        P = len(graphs)

        def load(plan):
            rows = plan.stage_indices([ix for seed in idx for ix in seed])
            gather_seeds_into(buffers, [rows[k * P:(k + 1) * P] for k in range(self.n_seeds)], plan.obs, plan.act, plan.nobs,
                              plan.rew, plan.done, idx_dev=plan.i_dev)
            return plan.load_noise(flat_noises)

        return self._run_update(tb, None, it, None, loader=load, per_morphology=per_morphology)

    def _check_seed_morphologies(self, parts_per_seed, what: str):
        """One list of (graph_dict, data) per seed, 1..MAX_PACKED_PARTS of them, the same morphologies in the same order for
        every seed.  Returns seed 0's graph dicts, which build the packed tables."""
        from .buffer import MAX_PACKED_PARTS
        self._check_list(parts_per_seed, what)
        first = parts_per_seed[0]
        if not 1 <= len(first) <= MAX_PACKED_PARTS:
            raise ValueError(f"{what}: a packed update holds 1 to {MAX_PACKED_PARTS} morphologies per seed, got {len(first)}")
        shape = [tuple(int(x) for x in g["parents"]) for g, _ in first]
        for k, parts in enumerate(parts_per_seed):
            if len(parts) != len(first):
                raise ValueError(f"{what}: seed {k} has {len(parts)} morphologies, seed 0 has {len(first)}")
            for i, (g, _) in enumerate(parts):
                if tuple(int(x) for x in g["parents"]) != shape[i]:
                    raise ValueError(f"{what}: seed {k} morphology {i} has other parents than seed 0's morphology {i}: every seed "
                                     f"needs the same morphologies in the same order")
        return [g for g, _ in first]

    def _seed_noises(self, noises, P: int):
        """None, or K lists of P noise tensors -> the seed-major flat list a packed plan takes."""
        if noises is None:
            return None
        self._check_list(noises, "noises")
        for k, nz in enumerate(noises):
            if len(nz) != P:
                raise ValueError(f"noises: seed {k} has {len(nz)} tensors for {P} morphologies")
        return [n for nz in noises for n in nz]

    # ------------------------------------------------------------------ acting
    @torch.no_grad()
    def select_actions(self, obs_per_seed, graphs, deterministic=False):
        """``Agent.select_actions`` for every seed in ONE replayed actor forward: obs_per_seed[k][i] is env i of seed k (its
        un-padded (41*N_i,) observation), graphs[i] env i's graph dict, the same list for every seed.  Returns per seed the
        list of (1, 3*N_i) numpy actions in env order."""
        self._check_list(obs_per_seed, "obs_per_seed")
        n = len(graphs)
        if n == 0 or any(len(o) != n for o in obs_per_seed):
            raise ValueError("select_actions needs, for every seed, one observation per graph")
        out = self._rollout_plan(self._rollout_tables_for(graphs)).run([o for seed in obs_per_seed for o in seed])
        return [[o.reshape(1, -1).copy() for o in out[k * n:(k + 1) * n]] for k in range(self.n_seeds)]

    def _check_list(self, xs, what: str):
        if len(xs) != self.n_seeds:
            raise ValueError(f"{what}: expected one per seed ({self.n_seeds}), got {len(xs)}")

    # single-agent entry points that have no seed-batched meaning here
    def _single(self, *a, **kw):
        raise NotImplementedError("SeedBatchedAgent steps every seed at once: use update / update_from_buffers / "
                                  "update_packed_per_seed / update_packed_from_buffers_per_seed / select_actions, or agent(k) for one seed")

    update_packed = update_packed_from_buffers = update_from_buffer = select_action = _single


# Per-seed hyper-parameters, as returned by get_hparams.  SeedBatchedAgent(args, seeds, hparams) and set_hparams also take
# `lr`, which sets both learning rates (the reference's single args.lr); a more specific key given with it wins.
HPARAM_KEYS = ("actor_lr", "critic_lr", "discount", "policy_noise", "noise_clip", "grad_clipping_value", "target_smoothing_tau",
               "reward_scale")
# args keys every seed shares: the delayed-update period, the action bound, the batch size and the architecture
SHARED_KEYS = ("policy_freq", "max_action", "batch_size", "actor_type", "critic_type", "limb_obs_size", "limb_action_size", "msg_dim",
               "max_children", "disable_fold", "td", "bu", "attention_embedding_size", "attention_heads", "attention_hidden_size",
               "attention_layers", "dropout_rate", "condition_decoder_on_features", "transformer_norm", "traversal_types", "rel_size")
_NON_NEGATIVE = ("lr", "actor_lr", "critic_lr", "grad_clipping_value", "policy_noise", "noise_clip")


def check_hparams(values: Dict, where: str) -> Dict[str, float]:
    """A dict of per-seed overrides -> {HPARAM_KEYS key: float}.  ValueError, in this order: a key every seed shares, an unknown
    key, a value that is not a finite real number, a negative learning rate, clip, policy noise or noise clip, and a tau
    outside [0, 1]."""
    if not isinstance(values, dict):
        raise ValueError(f"{where}: expected a dict of hyper-parameters, got {type(values).__name__}")
    for key in values:
        if key in SHARED_KEYS:
            raise ValueError(f"{where}: {key!r} is shared by every seed of a SeedBatchedAgent; set it in args")
    for key in values:
        if key != "lr" and key not in HPARAM_KEYS:
            raise ValueError(f"{where}: unknown hyper-parameter {key!r}; per-seed keys are lr, {', '.join(HPARAM_KEYS)}")
    for key, v in values.items():
        if isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(float(v)):
            raise ValueError(f"{where}: {key} must be a finite real number, got {v!r}")
    for key, v in values.items():
        if key in _NON_NEGATIVE and v < 0:
            raise ValueError(f"{where}: {key} must be >= 0, got {v}")
        if key == "target_smoothing_tau" and not 0.0 <= v <= 1.0:
            raise ValueError(f"{where}: target_smoothing_tau must lie in [0, 1], got {v}")
    out = {}
    if "lr" in values:
        out["actor_lr"] = out["critic_lr"] = float(values["lr"])
    out.update({k: float(v) for k, v in values.items() if k != "lr"})
    return out


def args_hparams(args) -> Dict[str, float]:
    """The HPARAM_KEYS values an ``Agent(args)`` trains with."""
    return dict(actor_lr=float(args.lr), critic_lr=float(args.lr), discount=float(args.discount), policy_noise=float(args.policy_noise),
                noise_clip=float(args.noise_clip), grad_clipping_value=float(args.grad_clipping_value),
                target_smoothing_tau=float(args.agent.target_smoothing_tau), reward_scale=float(args.agent.reward_scale))


def args_with(args, h: Dict[str, float]):
    """A copy of args (and of args.agent) holding the per-seed values h; args.lr only when both learning rates agree."""
    out = copy.copy(args)
    out.agent = copy.copy(args.agent)
    for key in ("discount", "policy_noise", "noise_clip", "grad_clipping_value"):
        setattr(out, key, h[key])
    out.agent.target_smoothing_tau, out.agent.reward_scale = h["target_smoothing_tau"], h["reward_scale"]
    if h["actor_lr"] == h["critic_lr"]:
        out.lr = h["actor_lr"]
    return out


def _check_count(K: int):
    if not 1 <= K <= MAX_SEEDS:
        raise ValueError(f"a seed-batched agent trains 1 to {MAX_SEEDS} seeds, got {K}")
