"""Helpers for the -m gpu parity tests (CUDA path through the C ABI vs the oracle)."""
import torch

from oracle import ref_loader, set_oracle as O
import parity


def make_modules(seed=parity.WEIGHT_SEED, use_tc=1):
    from sgrl_b200.modules import SEPolicy, SECritic
    args = ref_loader.default_args()
    actor = SEPolicy(41, 3, 32, 100, 1.0, None, False, False, False, args)
    critic = SECritic(41, 3, 32, 100, None, False, False, False, args)
    pa = {"actor." + k: v for k, v in O.synth_params("actor", seed).items()}
    pc = {"critic1." + k: v for k, v in O.synth_params("critic", seed + 1).items()}
    pc.update({"critic2." + k: v for k, v in O.synth_params("critic", seed + 2).items()})
    actor.load_state_dict(pa)
    critic.load_state_dict(pc)
    actor.use_tc = critic.use_tc = use_tc
    return actor, critic, pa, pc


def gemm_desc(persist, **pr):
    """One problem through sgrl_gemm_desc on the tcgen05 3xTF32 path, the planner's model everywhere but the persist override
    (0 | 1).  pr: SgrlGemmProblem fields (tensors for pointers; alpha, colscale, splitk, nb default to 1).  Returns the plan the
    library reports for the problem."""
    import ctypes
    from sgrl_b200._lib import GEMM_PLAN_FIELDS, GemmDesc, GemmPlanInfo, lib, ptr, stream, check
    d = GemmDesc()
    d.n, d.use_tc, d.persist = 1, 1, persist
    for f in ("bn", "split", "csk", "sm2", "tma_store", "group"):
        setattr(d, f, -1)
    p = d.pr[0]
    p.alpha, p.colscale, p.splitk, p.nb = 1.0, 1.0, 1, 1
    for k, v in pr.items():
        setattr(p, k, ptr(v) if torch.is_tensor(v) or v is None else v)
    info = GemmPlanInfo()
    check(lib.sgrl_gemm_desc(ctypes.byref(d), ctypes.byref(info), stream()), "sgrl_gemm_desc")
    torch.cuda.synchronize()
    return {f: getattr(info.pr[0], f) for f in GEMM_PLAN_FIELDS}


def to_cuda(d):
    return {k: (v.cuda() if torch.is_tensor(v) else [t.cuda() for t in v] if isinstance(v, list) and v and torch.is_tensor(v[0]) else v) for k, v in d.items()}


def stash_view(mod, stash, tb, nb, z, name, layer=-1, keep=1):
    """(T, per_token) view of a named stash buffer of net instance z."""
    from sgrl_b200 import _lib
    off, per = _lib.stash_info(mod._kind, mod._n_layers, tb.T, keep, name, layer)
    stride = stash.numel() // nb
    return stash[z * stride + off: z * stride + off + per * tb.T].view(tb.T, per)


def compare_stash(mod, stash, tb, nb, z, trace, n_layers=3, tol=2e-5, skip=()):
    """Return [(name, rel_err)] of every traced intermediate vs the CUDA stash."""
    out = []
    for key, ref in trace.items():
        if "." in key:
            l, name = key.split(".")
            l = int(l)
        else:
            l, name = -1, key
        if name in skip:
            continue
        got = stash_view(mod, stash, tb, nb, z, name, l)
        ref = ref.detach()
        if name == "P":     # (B,N,H,N) -> (T,H,16) zero padded
            B, N = ref.shape[0], ref.shape[1]
            pad = torch.zeros(B, N, 2, 16, device=ref.device, dtype=ref.dtype)
            pad[..., :N] = ref
            ref = pad
        if name in ("G1", "G2", "GH"):   # the kernels keep vec(G) as its packed upper triangle (sgrl_b200/packing.py) padded to 544
            from sgrl_b200.packing import pack_indices
            slots, ri, ci = pack_indices()
            full = ref.reshape(-1, 32, 32)
            ref = torch.zeros(full.shape[0], 544, device=ref.device, dtype=ref.dtype)
            ref[:, slots] = full[:, ri, ci]
        ref = ref.reshape(tb.T, -1).to(got.device)
        assert ref.shape == got.shape, (key, ref.shape, got.shape)
        out.append((key, parity.rel_err(got, ref)))
    return out


def relu_masks(mod, stash, tb, nb, z, n_layers=3):
    """Activation pattern of net instance z in a keep=True stash, keyed like the oracle's relu sites (set_oracle._relu)."""
    from sgrl_b200._lib import ACTOR
    mk = {}
    for l in range(n_layers):
        mk[f"{l}.A1"] = stash_view(mod, stash, tb, nb, z, "A1", l) > 0
        mk[f"{l}.A2"] = stash_view(mod, stash, tb, nb, z, "A2", l) > 0
        t31 = stash_view(mod, stash, tb, nb, z, "T31", l)
        mk[f"{l}.T3"], mk[f"{l}.T1"] = t31[:, :256] > 0, t31[:, 256:] > 0
    mk["AH"] = stash_view(mod, stash, tb, nb, z, "AH") > 0
    mk["BH"] = stash_view(mod, stash, tb, nb, z, "BH") > 0
    if mod._kind == ACTOR:
        mk["M1"] = stash_view(mod, stash, tb, nb, z, "M1") > 0
    return mk


def relu_flips(mod, stash, tb, nb, z, trace, prefix=""):
    """relu units that the CUDA forward and the oracle trace put on different sides of zero:
    [(site, |activation| / largest activation of the unit's row)] — ~1e-8 for a unit sitting on its kink."""
    out = []
    for key, ref in trace.items():
        l, nm = (int(key.split(".")[0]), key.split(".")[1]) if "." in key else (-1, key)
        if nm not in ("A1", "A2", "T31", "AH", "BH", "M1"):
            continue
        got = stash_view(mod, stash, tb, nb, z, nm, l)
        ref = ref.detach().reshape(tb.T, -1).to(got.device)
        for t, c in torch.nonzero((got > 0) != (ref > 0)).tolist():
            mag = max(abs(got[t, c].item()), abs(ref[t, c].item()))
            out.append((prefix + key, mag / max(ref[t].abs().max().item(), 1e-300)))
    return out
