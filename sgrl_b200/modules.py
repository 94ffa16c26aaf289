"""Drop-in SET modules: same class names, constructor signatures, ``forward`` contracts,
``change_morphology`` protocol and ``state_dict`` keys as the reference's
``SEActor.SEPolicy`` (src/SEActor.py:290-356) and ``SECritic.SECritic``
(src/SECritic.py:8-124) — the math runs in hand-written sm_100a kernels behind the C ABI
of ``include/sgrl_b200.h``.

Every reference tensor (SURVEY.md Appendix B, incl. the dead nn.MultiheadAttention
leftovers) is an ordinary ``nn.Parameter`` whose storage is a view into ONE flat fp32
arena per module, laid out by the library (csrc/layout.h).  Checkpoints load with
``load_state_dict``; kernels, Adam, Polyak and the gradient all-reduce stream the arena.
"""
from __future__ import annotations

import ctypes as C
import math
import operator
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib
from ._lib import ACTOR, CRITIC, NetCall, check, lib, ptr, stream

LIMB_OBS = 41
LIMB_ACT = 3
MAX_NODE = 15
USE_TC_DEFAULT = 1   # tcgen05 3xTF32 projections; 0 = fp32 SIMT everywhere


class _Holder(nn.Module):
    """Plain container used to reproduce the reference's dotted parameter names."""


def _device_default():
    return torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")


def _check_args(args):
    want = dict(attention_embedding_size=128, attention_heads=2, attention_hidden_size=256, rel_size=3)
    for k, v in want.items():
        got = getattr(args, k)
        if got != v:
            raise NotImplementedError(
                f"sgrl_b200 implements the reference SET hot path as shipped ({k}={v}); got {k}={got}. "
                "(The reference itself only works with 2 heads: subequivariant_attentions.py:117-118.)")
    if len(args.traversal_types) != 3:
        raise NotImplementedError("exactly the 3 traversal types ['pre','inlcrs','postlcrs'] are supported (main.py:54)")
    if not args.transformer_norm:
        raise NotImplementedError("transformer_norm=0 is not supported (start.sh uses 1)")
    if not (1 <= args.attention_layers <= 8):
        raise NotImplementedError("attention_layers must be in 1..8")


class GraphTables:
    """Device-side tables of one morphology (or of a packed mix of morphologies)."""

    def __init__(self, cu_limbs, rank3, tok_graph, relation, rel_off, T, G, tok_weight=None, parts=None, part_table=None):
        self.cu_limbs, self.rank3, self.tok_graph = cu_limbs, rank3, tok_graph
        self.relation, self.rel_off, self.T, self.G = relation, rel_off, T, G
        self.tok_weight = tok_weight          # (T) loss weight per token, packed mixed-morphology batches only
        self.parts = parts or [(0, T, 0, G, T // max(G, 1))]     # per morphology: (token0, token1, graph0, graph1, limbs)
        self.part_table = part_table          # (P,4) int32 {token0, token1, graph0, graph1} of self.parts, packed batches only
        self.nmax = max(p[4] for p in self.parts)                 # largest graph: sizes the attention kernel's staging


def make_tables(graph: Dict, batch: int, device) -> GraphTables:
    """Tables for `batch` graphs of one morphology (tokens packed sample-major, limb-minor,
    i.e. exactly the (B, N*41) row-major layout the reference feeds, SEActor.py:337-339)."""
    if "traversals" not in graph:
        raise ValueError("single-limb morphologies have no traversals/relation (utils.py:452-453); the SET net cannot run on them")
    n = len(graph["parents"])
    if n > 16 or n < 2:
        raise ValueError(f"{n} limbs: the SET kernels support 2..16 limbs per graph (positional tables hold 15)")
    ranks = torch.stack([t.to(torch.int32) for t in graph["traversals"]], dim=1).to(device)      # (N,3)
    if int(ranks.max()) >= MAX_NODE:
        raise ValueError("traversal rank exceeds the 15-row positional tables (SEActor.py:19)")
    rel = graph["relation"].to(device=device, dtype=torch.float32).contiguous()
    assert rel.shape == (n, n, 3), rel.shape
    cu = torch.arange(0, (batch + 1) * n, n, dtype=torch.int32, device=device)
    rank3 = ranks.repeat(batch, 1).contiguous()
    tok_graph = torch.arange(batch, dtype=torch.int32, device=device).repeat_interleave(n).contiguous()
    return GraphTables(cu, rank3, tok_graph, rel, None, batch * n, batch)


def make_packed_tables(parts, device, morph_count: Optional[float] = None) -> GraphTables:
    """Tables for a PACKED batch of several morphologies: parts = [(graph_dict, batch_i), ...].  Tokens are ordered
    morphology by morphology, sample-major, limb-minor; `cu_limbs` holds the ragged graph boundaries, `rel_off` each graph's
    offset into the concatenated relation tables, `tok_weight` = 1 / (#morphologies * B_i * N_i): the loss of the packed
    batch is the mean over morphologies of the reference's per-morphology loss (the reference steps the morphologies one
    after the other, src/trainer.py:245-250; SURVEY.md §8f rank 1).  morph_count (default: len(parts)) replaces
    #morphologies in the weight: a data-parallel rank that holds n_r of n morphologies passes n / world, so that the
    all-reduced sum / world is the mean over ALL n morphologies whatever the split (bench.py --set, N > 1).
    `part_table` holds each morphology's token and graph span for the per-morphology statistics (sgrl_td3_part_stats)."""
    cu, rank3, tokg, rel, reloff, w, spans = [0], [], [], [], [], [], []
    t0 = g0 = ro = 0
    m = len(parts)
    mw = float(morph_count) if morph_count else float(m)
    for graph, batch in parts:
        one = make_tables(graph, batch, "cpu")
        n = len(graph["parents"])
        cu.extend((one.cu_limbs[1:] + t0).tolist())
        rank3.append(one.rank3)
        tokg.append(one.tok_graph + g0)
        rel.append(one.relation.reshape(-1))
        reloff.extend([ro] * batch)
        w.append(torch.full((batch * n,), 1.0 / (mw * batch * n), dtype=torch.float32))
        spans.append((t0, t0 + batch * n, g0, g0 + batch, n))
        t0 += batch * n; g0 += batch; ro += n * n * 3
    i32 = lambda x: torch.as_tensor(x, dtype=torch.int32).to(device).contiguous()
    return GraphTables(i32(cu), torch.cat(rank3).to(device).contiguous(), torch.cat(tokg).to(torch.int32).to(device).contiguous(),
                       torch.cat(rel).to(device).contiguous(), i32(reloff), t0, g0,
                       tok_weight=torch.cat(w).to(device).contiguous() if (m > 1 or mw != 1.0) else None, parts=spans,
                       part_table=i32([s[:4] for s in spans]))


_VERSION_OF = operator.attrgetter("_version")


class SetNetModule(nn.Module):
    """nb reference ``TransformerModel``s (SEActor.py:170-287) in one flat arena."""

    def __init__(self, kind: int, net_names: List[str], args, max_action: float = 1.0, device=None):
        super().__init__()
        _check_args(args)
        self._kind = kind
        self._net_names = list(net_names)
        self._nb = len(net_names)
        self._n_layers = int(args.attention_layers)
        self._max_action = float(max_action)
        self._table = _lib.param_table(kind, self._n_layers)
        self._live, self._dead = _lib.arena_floats(kind, self._n_layers)
        self.use_tc = USE_TC_DEFAULT
        self._tables_cache: Dict = {}
        self._build(device or _device_default())
        # whatever a load wrote (also through a parent module's load_state_dict), the split is re-derived afterwards
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.invalidate_split())

    # ------------------------------------------------------------------ arena
    def _abs_offset(self, z: int, off: int, live: bool) -> int:
        return z * self._live + off if live else self._nb * self._live + z * self._dead + off

    def _build(self, device):
        total = self._nb * (self._live + self._dead)
        arena = torch.zeros(total, dtype=torch.float32, device=device)
        self._slots: List[Tuple[nn.Parameter, int, int]] = []
        for z, net in enumerate(self._net_names):
            root = _Holder()
            self.add_module(net, root)
            # register in the reference's state_dict order
            for name, shape, off, live in self._ordered_table():
                a = self._abs_offset(z, off, live)
                n = int(math.prod(shape))
                p = nn.Parameter(arena[a:a + n].view(shape), requires_grad=live)
                self._init_param(name, p.data)
                node = root
                parts = name.split(".")
                for part in parts[:-1]:
                    if not hasattr(node, part):
                        node.add_module(part, _Holder())
                    node = getattr(node, part)
                node.register_parameter(parts[-1], p)
                self._slots.append((p, a, n))
        self._arena = arena
        self._plist = [p for p, _, _ in self._slots]
        self._shared_counter = True                    # the parameters are views created from the arena: one version counter
        self._garena: Optional[torch.Tensor] = None
        self._split: Optional[torch.Tensor] = None     # (2, nb*live): tf32 hi / lo parts of the live arena
        self._split_fresh = False                      # True only while the agent's fused kernels keep it in sync
        self._anchor = torch.zeros((), device=device, requires_grad=True)

    def _ordered_table(self):
        """Library table re-ordered to the reference's registration order (cosmetic: keeps
        state_dict()/parameters() iteration identical to SEActor.py's)."""
        from .names import reference_order
        order = {n: i for i, n in enumerate(reference_order("actor" if self._kind == ACTOR else "critic", self._n_layers))}
        return sorted(self._table, key=lambda r: order[r[0]])

    @staticmethod
    def _init_param(name: str, t: torch.Tensor):
        """Same init distributions as the reference modules (nn.Linear / nn.Embedding /
        nn.LayerNorm / nn.MultiheadAttention defaults; SEActor.py:232-235 for the encoders)."""
        with torch.no_grad():
            if "embeddings" in name:
                t.normal_(0, 1)
            elif "norm" in name:
                t.fill_(1.0 if name.endswith("weight") else 0.0)
            elif name in ("encoder.weight", "g_encoder.weight"):
                t.uniform_(-0.1, 0.1)
            elif name.endswith("in_proj_weight"):
                nn.init.xavier_uniform_(t)
            elif name.endswith("in_proj_bias") or name.endswith("out_proj.bias"):
                t.zero_()
            elif t.dim() == 2:
                nn.init.kaiming_uniform_(t, a=math.sqrt(5))
            else:
                t.zero_()   # biases are filled after their weights below

    def _init_biases(self):
        sd = dict(self.named_parameters())
        with torch.no_grad():
            for k, b in sd.items():
                if k.endswith(".bias") and "norm" not in k and "in_proj" not in k and "out_proj" not in k:
                    w = sd[k[:-4] + "weight"]
                    bound = 1.0 / math.sqrt(w.shape[1])
                    b.uniform_(-bound, bound)

    def _apply(self, fn, recurse=True):
        super()._apply(fn, recurse)
        self._reflatten()
        return self

    def _reflatten(self):
        """Restore the flat-arena aliasing after .to()/.cuda()/.float() replaced parameter storage."""
        p0 = self._slots[0][0]
        dev = p0.device
        ok = self._arena.device == dev and all(p.data_ptr() == self._arena.data_ptr() + 4 * a for p, a, _ in self._slots)
        if ok:
            return
        arena = torch.zeros(self._arena.numel(), dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, a, n in self._slots:
                arena[a:a + n].copy_(p.data.reshape(-1).to(torch.float32))
                p.data = arena[a:a + n].view(p.shape)
                p.grad = None
        self._arena = arena
        self._shared_counter = False                   # p.data = ... keeps each parameter's own counter
        self._garena = None
        self._split, self._split_fresh = None, False
        self._anchor = torch.zeros((), device=dev, requires_grad=True)
        self._tables_cache.clear()

    @property
    def live_arena(self) -> torch.Tensor:
        """The nb*live_floats prefix the kernels, Adam and the all-reduce operate on."""
        return self._arena[: self._nb * self._live]

    @property
    def full_arena(self) -> torch.Tensor:
        return self._arena

    def grad_arena(self) -> torch.Tensor:
        if self._garena is None or self._garena.device != self._arena.device:
            self._garena = torch.zeros(self._nb * self._live, dtype=torch.float32, device=self._arena.device)
        return self._garena

    # ------------------------------------------------------------------ pre-split weights for the tcgen05 projections
    SPLIT_MIN_TOKENS = 64      # below this every projection is launch-bound: not worth a pass over the arena

    def split_arena(self) -> torch.Tensor:
        if self._split is None or self._split.device != self._arena.device:
            self._split = torch.empty(2, self._nb * self._live, dtype=torch.float32, device=self._arena.device)
            self._split_fresh = False
        return self._split

    def refresh_split(self):
        """hi = tf32(w), lo = tf32(w - hi) over the live arena (one streaming pass)."""
        sp = self.split_arena()
        check(lib.sgrl_split_tf32(ptr(self.live_arena), ptr(sp[0]), ptr(sp[1]), sp.shape[1], stream()), "sgrl_split_tf32")
        self.mark_split_fresh()

    def _write_stamp(self) -> int:
        """Sum of the version counters of the arena and of every parameter.  In-place torch writes (p.copy_, optimizers,
        load_state_dict) bump the counter of the tensor they go through: right after construction the parameters share
        the arena's counter, after a re-flatten (.to() / .cuda()) each parameter has its own, so all of them are summed.
        Writes through ``p.data`` / raw pointers bump nothing: callers that do that must call invalidate_split()."""
        if self._shared_counter:
            return self._arena._version
        return self._arena._version + sum(map(_VERSION_OF, self._plist))

    def mark_split_fresh(self):
        """Called after a kernel (split / fused Adam / Polyak) rewrote the split from the current arena contents."""
        self._split_fresh, self._split_version = True, self._write_stamp()

    def invalidate_split(self):
        """Force the next tcgen05 pass to re-derive the tf32 hi/lo split from the parameters.  Needed only after writes
        the version counters cannot see (``p.data.copy_(...)``, custom kernels writing the arena)."""
        self._split_fresh = False

    def split_is_fresh(self) -> bool:
        return self._split is not None and self._split_fresh and self._split_version == self._write_stamp()

    def _split_for(self, T: int, trusted: bool):
        """(hi, lo) to hand to the kernels, or (None, None).  Only a caller that owns every write to the arena
        (Agent.update: fused Adam / Polyak keep the split in sync) may pass trusted=True; everyone else gets a
        split recomputed from the current parameter values, because nn.Parameters can be modified behind our back."""
        if not self.use_tc or T < self.SPLIT_MIN_TOKENS or self._arena.device.type != "cuda":
            return None, None
        if not (trusted and self.split_is_fresh()):
            self.refresh_split()
        return self._split[0], self._split[1]

    # ------------------------------------------------------------------ morphology protocol
    def change_morphology(self, graph):
        """SEActor.py:349-356 / SECritic.py:117-124."""
        self.graph = graph
        self.parents = graph["parents"]
        self.num_limbs = len(self.parents)
        self.msg_down = [None] * self.num_limbs
        self.msg_up = [None] * self.num_limbs
        self.action = [None] * self.num_limbs
        self.input_state = [None] * self.num_limbs

    def _tables(self, batch: int) -> GraphTables:
        g = self.graph
        key = (id(g.get("relation")), tuple(g["parents"]), batch)
        t = self._tables_cache.get(key)
        if t is None:
            if len(self._tables_cache) > 64:
                self._tables_cache.clear()
            t = make_tables(g, batch, self._arena.device)
            self._tables_cache[key] = t
        return t

    # ------------------------------------------------------------------ raw kernel passes
    def _call(self, tb: GraphTables, nb: int, keep: int, stash, grads=None, ws=None, split=(None, None), in_nets: int = 0) -> NetCall:
        k = NetCall()
        k.kind, k.n_layers, k.nb, k.T, k.G, k.in_nets = self._kind, self._n_layers, nb, tb.T, tb.G, in_nets
        k.keep, k.use_tc, k.max_limbs = keep, int(self.use_tc), int(tb.nmax)
        k.params = ptr(self.live_arena)
        k.params_hi, k.params_lo = ptr(split[0]), ptr(split[1])
        k.grads = ptr(grads)
        k.stash = ptr(stash)
        k.stash_stride = stash.numel() // nb
        if ws is not None:
            k.ws = ptr(ws)
            k.ws_stride = ws.numel() // nb
        k.cu_limbs, k.rel_off, k.relation, k.rank3 = ptr(tb.cu_limbs), ptr(tb.rel_off), ptr(tb.relation), ptr(tb.rank3)
        k.max_action = self._max_action
        return k

    def stash_floats(self, T: int, keep: bool, nb: int) -> int:
        return nb * lib.sgrl_stash_floats(self._kind, self._n_layers, T, int(keep))

    def ws_floats(self, T: int, nb: int) -> int:
        return nb * lib.sgrl_ws_floats(self._n_layers, T)

    def forward_raw(self, tb: GraphTables, obs: torch.Tensor, act: Optional[torch.Tensor], keep: bool, nb: Optional[int] = None,
                    out: Optional[torch.Tensor] = None, trusted_split: bool = False, stash: Optional[torch.Tensor] = None,
                    in_nets: int = 0):
        """Run nb nets on tokens obs (T,41) [act (T,3)].  Returns (out (nb,T,od), stash).  `out` / `stash` may be
        caller-owned buffers (Agent.update's static plan); otherwise they are allocated here.  in_nets = 0: every net reads
        the same obs / act; in_nets = K: obs (K*T,41) [act (K*T,3)] hold K input blocks and net z reads block z % K."""
        nb = self._nb if nb is None else nb
        od = 3 if self._kind == ACTOR else 1
        dev = self._arena.device
        if dev.type != "cuda":
            raise _lib.SgrlError("sgrl_b200 modules only run on CUDA devices (no CPU fallback)")
        if stash is None:
            stash = torch.empty(self.stash_floats(tb.T, keep, nb), dtype=torch.float32, device=dev)
        if out is None:
            out = torch.empty(nb, tb.T, od, dtype=torch.float32, device=dev)
        k = self._call(tb, nb, int(keep), stash, split=self._split_for(tb.T, trusted_split), in_nets=in_nets)
        blk = tb.T if in_nets else 0
        check(lib.sgrl_set_forward(C.byref(k), ptr(obs), blk * LIMB_OBS, ptr(act), blk * LIMB_ACT, ptr(out), tb.T * od, stream()),
              "sgrl_set_forward")
        return out, stash

    def backward_raw(self, tb: GraphTables, stash: torch.Tensor, dout: torch.Tensor, nb: int, grads: Optional[torch.Tensor],
                     want_dact: bool, trusted_split: bool = False, ws: Optional[torch.Tensor] = None, dact: Optional[torch.Tensor] = None,
                     dobs: Optional[torch.Tensor] = None):
        """dout (nb,T,od).  Accumulates parameter gradients into `grads` (None: data-only).  `dobs`: optional caller-owned
        contiguous (nb,T,41) fp32 CUDA tensor that receives the gradient w.r.t. the observation input (overwritten)."""
        dev = self._arena.device
        if ws is None:
            ws = torch.empty(self.ws_floats(tb.T, nb), dtype=torch.float32, device=dev)
        if want_dact and dact is None:
            dact = torch.empty(nb, tb.T, 3, dtype=torch.float32, device=dev)
        if dobs is not None and (dobs.dtype != torch.float32 or not dobs.is_contiguous() or tuple(dobs.shape) != (nb, tb.T, LIMB_OBS)):
            raise ValueError(f"dobs must be a contiguous float32 ({nb}, {tb.T}, {LIMB_OBS}) tensor, got {dobs.dtype} {tuple(dobs.shape)}")
        od = 3 if self._kind == ACTOR else 1
        k = self._call(tb, nb, 1, stash, grads=grads, ws=ws, split=self._split_for(tb.T, trusted_split))
        check(lib.sgrl_set_backward_dobs(C.byref(k), ptr(dout), tb.T * od, 1 if grads is not None else 0, ptr(dact), tb.T * 3,
                                         ptr(dobs), tb.T * LIMB_OBS, stream()), "sgrl_set_backward_dobs")
        return dact

    # ------------------------------------------------------------------ autograd bridge
    def _run(self, state: torch.Tensor, action: Optional[torch.Tensor], nb: int) -> torch.Tensor:
        B = state.shape[0]
        tb = self._tables(B)
        obs = state.detach().to(torch.float32).contiguous()
        act = action.detach().to(torch.float32).contiguous() if action is not None else None
        state_grad = state.requires_grad
        needs = torch.is_grad_enabled() and (any(p.requires_grad for p, _, _ in self._slots) or (action is not None and action.requires_grad)
                                             or state_grad)
        if not needs:
            out, _ = self.forward_raw(tb, obs, act, keep=False, nb=nb)
            return out
        return _SetNetFn.apply(self, tb, nb, self._anchor, obs, action if action is not None and action.requires_grad else None, act,
                               state if state_grad else None)


class _SetNetFn(torch.autograd.Function):
    """loss.backward() support for the drop-in modules.  Parameter gradients are produced by
    the backward kernels into a scratch arena and then added to each ``p.grad`` (torch
    semantics: accumulate until zero_grad).  Gradients w.r.t. the action (critics) and the
    state come back through autograd like any torch input gradient."""

    @staticmethod
    def forward(ctx, mod: SetNetModule, tb, nb, anchor, obs, action_in, act, state_in=None):
        out, stash = mod.forward_raw(tb, obs, act, keep=True, nb=nb)
        ctx.mod, ctx.tb, ctx.nb, ctx.stash = mod, tb, nb, stash
        ctx.want_dact = action_in is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        mod, nb = ctx.mod, ctx.nb
        want_w = any(p.requires_grad for p, _, _ in mod._slots)
        want_dobs = ctx.needs_input_grad[7]
        scratch = torch.zeros(mod._nb * mod._live, dtype=torch.float32, device=dout.device) if want_w else None
        dobs = torch.empty(nb, ctx.tb.T, LIMB_OBS, dtype=torch.float32, device=dout.device) if want_dobs else None
        dact = mod.backward_raw(ctx.tb, ctx.stash, dout.contiguous().to(torch.float32), nb, scratch, ctx.want_dact, dobs=dobs)
        if want_w:
            for p, a, n in mod._slots:
                if not p.requires_grad or a >= nb * mod._live:
                    continue   # dead tensors and nets that did not run (Q1 uses critic1 only) get no gradient
                g = scratch[a:a + n].view(p.shape)
                if p.grad is None:
                    p.grad = g          # views of this call's private scratch arena
                else:
                    p.grad = p.grad + g
        ctx.stash = None
        d_action = None
        if ctx.want_dact:
            d_action = dact.sum(0).view(ctx.tb.G, -1)
        d_state = dobs.sum(0).view(ctx.tb.G, -1) if want_dobs else None      # twin critics: sum over both nets, like d_action
        return None, None, None, None, None, d_action, None, d_state


class SEPolicy(SetNetModule):
    """Drop-in for SEActor.SEPolicy (src/SEActor.py:290-356)."""

    def __init__(self, state_dim, action_dim, msg_dim, batch_size, max_action, max_children, disable_fold, td, bu, args=None):
        if state_dim != LIMB_OBS or action_dim != LIMB_ACT:
            raise NotImplementedError("the SET hot path is defined for 41-float limb observations and 3 actions per limb")
        super().__init__(ACTOR, ["actor"], args, max_action=max_action)
        self._init_biases()
        self.num_limbs = 1
        self.msg_down = [None]; self.msg_up = [None]; self.action = [None]; self.input_state = [None]
        self.max_action = max_action
        self.msg_dim, self.batch_size, self.max_children, self.disable_fold = msg_dim, batch_size, max_children, disable_fold
        self.state_dim, self.action_dim = state_dim, action_dim

    def forward(self, state, mode="train"):
        """state (B, N*41) -> max_action*tanh(actions) (B, N*3); SEActor.py:334-347."""
        self.clear_buffer()
        B = state.shape[0]
        if state.shape[1] != self.state_dim * self.num_limbs:
            raise RuntimeError(f"shape '[{B}, {self.num_limbs}, -1]' is invalid for input of size {state.numel()}")
        out = self._run(state, None, 1)
        self.action = out[0].reshape(B, self.num_limbs * self.action_dim)
        return self.action

    def clear_buffer(self):
        """ModularActor.py:351-358."""
        self.msg_down = [None] * self.num_limbs
        self.msg_up = [None] * self.num_limbs
        self.action = [None] * self.num_limbs
        self.input_state = [None] * self.num_limbs
        self.zeroFold_td = None
        self.zeroFold_bu = None
        self.fold = None


class SECritic(SetNetModule):
    """Drop-in for SECritic.SECritic (src/SECritic.py:8-124): twin per-limb Q networks."""

    def __init__(self, state_dim, action_dim, msg_dim, batch_size, max_children, disable_fold, td, bu, args=None):
        if state_dim != LIMB_OBS or action_dim != LIMB_ACT:
            raise NotImplementedError("the SET hot path is defined for 41-float limb observations and 3 actions per limb")
        super().__init__(CRITIC, ["critic1", "critic2"], args)
        self._init_biases()
        self.num_limbs = 1
        self.x1 = [None]; self.x2 = [None]; self.input_state = [None]; self.input_action = [None]
        self.msg_down = [None]; self.msg_up = [None]
        self.msg_dim, self.batch_size, self.max_children, self.disable_fold = msg_dim, batch_size, max_children, disable_fold
        self.state_dim, self.action_dim = state_dim, action_dim

    def _check(self, state):
        assert (
            state.shape[1] == self.state_dim * self.num_limbs
        ), "state.shape[1] expects {} but got {} with num_limbs being {} and state_dim being {}".format(
            self.state_dim * self.num_limbs, state.shape[1], self.num_limbs, self.state_dim)

    def forward(self, state, action):
        """(B,N*41),(B,N*3) -> (Q1 (B,N), Q2 (B,N)); SECritic.py:66-91."""
        self.clear_buffer()
        self._check(state)
        out = self._run(state, action, 2)
        B = state.shape[0]
        self.x1, self.x2 = out[0].reshape(B, self.num_limbs), out[1].reshape(B, self.num_limbs)
        return self.x1, self.x2

    def Q1(self, state, action):
        """critic1 only; SECritic.py:93-104."""
        self.clear_buffer()
        out = self._run(state, action, 1)
        self.x1 = out[0].reshape(state.shape[0], self.num_limbs)
        return self.x1

    def clear_buffer(self):
        """SECritic.py:106-115."""
        self.x1 = [None] * self.num_limbs
        self.x2 = [None] * self.num_limbs
        self.input_state = [None] * self.num_limbs
        self.input_action = [None] * self.num_limbs
        self.msg_down = [None] * self.num_limbs
        self.msg_up = [None] * self.num_limbs
        self.zeroFold_td = None
        self.zeroFold_bu = None
        self.fold = None
