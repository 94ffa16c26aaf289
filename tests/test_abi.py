"""CPU-side checks of the C-ABI library: it loads without a GPU, exports every symbol that
include/sgrl_b200.h declares, and its parameter table reproduces the reference state_dict."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import set_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "sgrl_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sgrl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol():
    from sgrl_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(_lib.lib, s), f"{s} declared in include/sgrl_b200.h but not exported"
    assert set(_lib.EXPORTS) == set(syms), set(_lib.EXPORTS) ^ set(syms)
    assert _lib.lib.sgrl_version() >= 2


@pytest.mark.parametrize("kind,kname", [(0, "actor"), (1, "critic")])
def test_param_table_matches_reference_inventory(kind, kname):
    from sgrl_b200 import _lib
    table = _lib.param_table(kind, 3)
    spec = dict(O.param_spec(kname))
    assert {n for n, _, _, _ in table} == set(spec)
    live, dead = _lib.arena_floats(kind, 3)
    spans = {True: [], False: []}
    for n, shape, off, is_live in table:
        assert tuple(shape) == spec[n], n
        assert is_live == (not O.is_dead(n))
        assert off % 16 == 0
        spans[is_live].append((off, off + int(np.prod(shape))))
    for is_live, cap in ((True, live), (False, dead)):
        s = sorted(spans[is_live])
        assert all(a[1] <= b[0] for a, b in zip(s, s[1:])), "overlapping tensors"
        assert s[-1][1] <= cap
    offs = {n: off for n, _, off, _ in table}
    for l in range(3):
        p = f"transformer_encoder.layers.{l}."
        # stacked operands must be adjacent: q|k|v and linear3|linear1
        assert offs[p + "self_attn.k_proj.weight"] - offs[p + "self_attn.q_proj.weight"] == 65536
        assert offs[p + "self_attn.v_proj.weight"] - offs[p + "self_attn.k_proj.weight"] == 65536
        assert offs[p + "self_attn.v_proj.bias"] - offs[p + "self_attn.q_proj.bias"] == 512
        assert offs[p + "linear1.weight"] - offs[p + "linear3.weight"] == 65536
        assert offs[p + "linear1.bias"] - offs[p + "linear3.bias"] == 256


def test_error_reporting_without_gpu():
    from sgrl_b200 import _lib
    assert _lib.lib.sgrl_param_count(7, 3) < 0
    assert b"bad kind" in _lib.lib.sgrl_last_error()
    assert _lib.lib.sgrl_stash_floats(0, 3, 900, 1) > _lib.lib.sgrl_stash_floats(0, 3, 900, 0) > 0
    assert _lib.lib.sgrl_ws_floats(3, 900) > 0


def test_attention_bwd_rejects_drel_w_without_relation():
    """The backward forms d rel_encoder.weight from the relation tables: drel_w without relation is refused before any
    launch (G = 0: even without the check nothing would be enqueued, so the call cannot touch memory)."""
    from sgrl_b200 import _lib
    lib, fake = _lib.lib, 256
    rc = lib.sgrl_attention_bwd(fake, fake, fake, fake, fake, fake, fake, None, None, 0, 0, fake, fake, fake, None)
    assert rc < 0 and b"drel_w needs relation" in lib.sgrl_last_error()


def test_deterministic_mode_switch_without_gpu():
    """sgrl_deterministic(enable): 1 / 0 switch the mode, -1 only queries; each call returns the previous state (no GPU work)."""
    from sgrl_b200 import _lib
    lib = _lib.lib
    prev = lib.sgrl_deterministic(-1)
    assert prev in (0, 1)
    assert lib.sgrl_deterministic(1) == prev and lib.sgrl_deterministic(-1) == 1
    assert lib.sgrl_deterministic(0) == 1 and lib.sgrl_deterministic(-1) == 0
    lib.sgrl_deterministic(prev)


def test_modules_build_on_cpu_with_reference_state_dict_keys():
    import torch
    from oracle import ref_loader
    from sgrl_b200.modules import SEPolicy, SECritic
    args = ref_loader.default_args()
    a = SEPolicy(41, 3, 32, 100, 1.0, None, False, False, False, args)
    c = SECritic(41, 3, 32, 100, None, False, False, False, args)
    assert list(a.state_dict().keys()) == ["actor." + n for n, _ in O.param_spec("actor")]
    assert list(c.state_dict().keys()) == [f"critic{i}." + n for i in (1, 2) for n, _ in O.param_spec("critic")]
    assert sum(v.numel() for v in a.state_dict().values()) == 4712712
    assert sum(v.numel() for v in c.state_dict().values()) == 8761330
    # parameters alias one flat arena; load_state_dict writes through
    sd = {"actor." + k: v for k, v in O.synth_params("actor", 3).items()}
    a.load_state_dict(sd)
    k = "actor.transformer_encoder.layers.2.linear4.weight"
    p = dict(a.named_parameters())[k]
    assert p.data_ptr() >= a.full_arena.data_ptr() and torch.equal(p.data, sd[k].to(p.device))     # the arena is on cuda:0 when there is one
    assert abs(a.live_arena.double().sum().item() - sum(v.double().sum().item() for n, v in sd.items() if not O.is_dead(n))) < 1e-3
    a2 = a.double().float()      # _apply must restore the aliasing
    assert all(q.data_ptr() == a2.full_arena.data_ptr() + 4 * off for q, off, _ in a2._slots)
    if not torch.cuda.is_available():
        a.change_morphology({"parents": [-1, 0], "traversals": [torch.tensor([0, 1])] * 3, "relation": torch.zeros(2, 2, 3)})
        with pytest.raises(Exception, match="CUDA"):
            a(torch.zeros(1, 82))
    with pytest.raises(NotImplementedError):
        SEPolicy(41, 3, 32, 100, 1.0, None, False, False, False, ref_loader.default_args(attention_heads=4))


def _desc(**over):
    """A one-problem sgrl_gemm_desc descriptor on fake (never dereferenced) 16-byte aligned addresses: 2304 x 256 x 64, pre-split
    B, tcgen05 path, every planner override at -1 (the model)."""
    from sgrl_b200 import _lib
    d = _lib.GemmDesc()
    p = d.pr[0]
    p.A, p.lda, p.B, p.B_hi, p.B_lo, p.ldb, p.C, p.ldc = 1 << 20, 64, 2 << 20, 3 << 20, 4 << 20, 64, 5 << 20, 256
    p.M, p.N, p.K, p.alpha, p.colscale, p.splitk, p.nb = 2304, 256, 64, 1.0, 1.0, 1, 1
    d.n, d.use_tc = 1, 1
    for f in ("bn", "split", "csk", "sm2", "persist", "tma_store", "group"):
        setattr(d, f, -1)
    for k, v in over.items():
        setattr(d if hasattr(d, k) else p, k, v)
    return d


@pytest.mark.parametrize("over,msg", [
    (dict(bias=6 << 20, splitk=4, accumulate=1), b"no bias"),                    # the atomic split-K epilogue carries no bias
    (dict(splitk=4, accumulate=0), b"accumulate = 1"),                           # partial sums are added into C
    (dict(csk=3), b"without k-blocks"),                                          # K = 64: 2 k-blocks for 3 ranks
    (dict(csk=1), b"csk override"),
    (dict(bn=96), b"bn override"),
    (dict(split=4), b"split override needs splitk > 1"),
    (dict(persist=1, rowsum=6 << 20), b"persistent kernels cannot"),
    (dict(tma_store=1, accumulate=1), b"TMA-store epilogue cannot"),
    (dict(sm2=1, trans_a=1, lda=2304), b"two-CTAs-per-SM variant cannot"),
    (dict(sm2=1, persist=1), b"exclude each other"),
    (dict(group=1), b"several problems"),
    (dict(use_tc=0, bn=64), b"need the tcgen05 path"),
    (dict(use_tc=0, rowsum=6 << 20), b"need the tcgen05 path"),
    (dict(n=5), b"1..4 problems"),
    (dict(B_lo=0), b"go together"),
    (dict(M=64, N=128, K=255), b"not eligible"),                                 # M N K < 2^21: launch-bound sizes stay on SIMT
])
def test_gemm_desc_refuses_invalid_descriptors(over, msg):
    """sgrl_gemm_desc refuses a descriptor its kernels cannot run, or an override the problem cannot take, before anything is
    enqueued (fake addresses: a call that got as far as a launch would fault, so a refusal is the only way to pass here)."""
    from sgrl_b200 import _lib
    lib = _lib.lib
    rc = lib.sgrl_gemm_desc(ctypes.byref(_desc(**over)), None, None)
    assert rc < 0 and msg in lib.sgrl_last_error(), lib.sgrl_last_error()


def test_gemm_refuses_bias_or_store_with_split_k():
    """splitk > 1 lets K be split with atomic adds into C: sgrl_gemm and sgrl_gemm_presplit refuse it with a bias or without
    accumulate, on both paths (the tcgen05 split epilogue used to drop the bias while the SIMT kernel added it)."""
    from sgrl_b200 import _lib
    lib, f = _lib.lib, 1 << 20
    for use_tc in (0, 1):
        assert lib.sgrl_gemm(f, 64, 1, f, 64, 1, f, 64, 30, 128, 2304, 1.0, f, None, 0, 1, 8, use_tc, None) < 0
        assert b"no bias" in lib.sgrl_last_error()
        assert lib.sgrl_gemm(f, 64, 1, f, 64, 1, f, 64, 30, 128, 2304, 1.0, None, None, 0, 0, 8, use_tc, None) < 0
        assert b"accumulate = 1" in lib.sgrl_last_error()
    assert lib.sgrl_gemm_presplit(f, 64, 1, f, f, 64, 1, f, 64, 30, 128, 2304, 1.0, f, None, 0, 1, 8, None) < 0
    assert b"no bias" in lib.sgrl_last_error()


_F = 1 << 20          # fake, never dereferenced, 16-byte aligned device addresses
_ARGS = {             # a valid call of each single-kernel entry point (ABI 11), argument by argument, grid and stream at the end
    "sgrl_embed_fwd": dict(obs=_F, zs_obs=0, act=None, zs_act=0, rank3=_F, Wg=_F, We=_F, be=_F, E0=_F, E1=_F, E2=_F, zs_p=0, V0=_F, GD=_F,
                           SH=_F, ldsh=145, VG=_F, H=_F, ldh=256, zs_s=0, T=100, ng=17, nb=2, in_nets=1),
    "sgrl_input_grad": dict(dvg0=_F, dh0=_F, dzh=_F, dzh2=_F, dsh=_F, ldsh=145, dz="dz", dog="dog", P="P", Wg=_F, We=_F, gg=_F, gph=_F, ng=17,
                            dout=_F, zs_do=0, out=_F, w3=_F, max_action=1.0, dobs=_F, zs_dobs=0, cu_limbs=_F, G=10, T=100, L=3, zs_w=0,
                            zs_s=0, zs_p=0, nb=1),
    "sgrl_pos_embed_bwd": dict(dH=_F, ldh=128, zs_w=0, rank3=_F, dE0=_F, dE1=_F, dE2=_F, zs_g=0, T=100, nb=1),
    "sgrl_layernorm_fwd": dict(a=_F, lda=256, b=None, ldb=0, gamma=_F, beta=_F, zs_p=0, x=_F, y=_F, ldy=145, y2=None, ldy2=0, stats=_F,
                               zs_s=0, T=100, nb=1),
    "sgrl_layernorm_bwd": dict(dy1=_F, ld1=128, dy2=None, ld2=0, x=_F, ldx=128, stats=_F, zs_s=0, gamma=_F, zs_p=0, dx=_F, lddx=128, zs_w=0,
                               dgamma=_F, dbeta=_F, zs_g=0, rd_y=None, rd_ldy=0, rd_F=None, rd_dF=None, rd_out=None, rd_ldout=0, T=100,
                               nb=1),
    "sgrl_matapply_fwd": dict(Z=_F, M=_F, R=_F, zs_s=0, T=100, nb=1),
    "sgrl_matapply_bwd": dict(dR=_F, Z=_F, M=_F, F=_F, zs_s=0, dZ=_F, dT=_F, dF=_F, zs_w=0, T=100, nb=1),
    "sgrl_matapply_l5_fwd": dict(Z=_F, M=_F, W5=_F, zs_p=0, Vg=_F, dV=_F, R=None, Vn=_F, zs_s=0, T=100, nb=1),
    "sgrl_matapply_l5_bwd": dict(dVn=_F, W5=_F, zs_p=0, Z=_F, M=_F, F=_F, zs_s=0, dZ=_F, dT=_F, dF=_F, zs_w=0, T=100, nb=1),
    "sgrl_actor_out_fwd": dict(R=_F, V0=_F, wd=_F, zs_p=0, W3=_F, out=_F, zs_s=0, max_action=1.0, T=100, nb=1),
    "sgrl_actor_out_bwd": dict(dout=_F, zs_do=0, out=_F, R=_F, V0=_F, zs_s=0, wd=_F, zs_p=0, dR=_F, zs_w=0, dwd=_F, zs_g=0, max_action=1.0,
                               T=100, nb=1),
    "sgrl_rowdiv_bwd": dict(dy=_F, lddy=768, zs_w=0, y=_F, ldy=768, F=_F, zs_s=0, dF=_F, N=768, colscale=0.5, cs_n=256, src=None, ldsrc=0,
                            zs_src=0, T=100, nb=1),
    "sgrl_colsum": dict(X=_F, ldx=128, zs_x=0, out=_F, zs_o=0, M=100, N=128, alpha=1.0, nb=1),
    "sgrl_block_copy": dict(dst=_F, ldd=3, zs_d=0, src=_F, lds=3, zs_src=0, src2=None, lds2=0, zs_src2=0, M=100, N=3, add=0, nb=1),
    "sgrl_fold_sym": dict(params=_F, zs_p=0, wf=_F, zs_s=0, plane=1024, with_split=1, src="src", dst="dst", rows="rows", n=7, nb=1),
    "sgrl_unfold_sym": dict(gf=_F, zs_w=0, grads=_F, zs_g=0, src="src", dst="dst", rows="rows", n=7, nb=1),
}


def _call(name, **over):
    from sgrl_b200 import _lib
    a = dict(_ARGS[name], **over)
    host = {"dz": (ctypes.c_void_p * 24)(*([_F] * 24)), "dog": (ctypes.c_void_p * 8)(*([_F] * 8)), "P": (ctypes.c_void_p * 8)(*([_F] * 8)),
            "src": (ctypes.c_int64 * 17)(*([0] * 17)), "dst": (ctypes.c_int64 * 17)(*([544 * 256 * i for i in range(17)])),
            "rows": (ctypes.c_int32 * 17)(*([256] * 17))}
    vals = [host[v] if isinstance(v, str) else v for v in a.values()]
    return getattr(_lib.lib, name)(*vals, None, None)


@pytest.mark.parametrize("name,over,msg", [
    ("sgrl_embed_fwd", dict(obs=None), b"null pointer"),
    ("sgrl_embed_fwd", dict(ng=18), b"ng must be 17"),
    ("sgrl_embed_fwd", dict(act=_F), b"act is read by critics"),                    # actor layout with an action
    ("sgrl_embed_fwd", dict(ng=20), b"act is read by critics"),                     # critic without one
    ("sgrl_embed_fwd", dict(nb=17), b"nb must be 1..16"),
    ("sgrl_embed_fwd", dict(nb=0), b"nb must be 1..16"),
    ("sgrl_embed_fwd", dict(in_nets=3), b"in_nets must be 1..nb"),
    ("sgrl_embed_fwd", dict(in_nets=0), b"in_nets must be 1..nb"),
    ("sgrl_embed_fwd", dict(T=-1), b"T must be >= 0"),
    ("sgrl_input_grad", dict(dobs=None), b"null pointer"),
    ("sgrl_input_grad", dict(L=0), b"L must be 1..8"),
    ("sgrl_input_grad", dict(L=9), b"L must be 1..8"),
    ("sgrl_input_grad", dict(ng=20), b"dzh2"),                                      # actor head with the critic's ng
    ("sgrl_input_grad", dict(dzh2=None), b"dzh2"),                                  # critic head with the actor's ng
    ("sgrl_input_grad", dict(ng=19, dzh2=None), b"ng must be 17"),
    ("sgrl_input_grad", dict(w3=None), b"needs gph, dout, out and w3"),
    ("sgrl_input_grad", dict(dog=None), b"null pointer"),
    ("sgrl_input_grad", dict(zs_w=3), b"8-byte aligned"),                           # float2 loads of d og
    ("sgrl_input_grad", dict(nb=17), b"nb must be 1..16"),
    ("sgrl_input_grad", dict(T=-5), b"T must be >= 0"),
    ("sgrl_pos_embed_bwd", dict(rank3=None), b"null pointer"),
    ("sgrl_pos_embed_bwd", dict(nb=0), b"nb must be 1..16"),
    ("sgrl_layernorm_fwd", dict(stats=None), b"null pointer"),
    ("sgrl_layernorm_fwd", dict(gamma=_F + 4), b"gamma, beta and zs_p"),
    ("sgrl_layernorm_fwd", dict(beta=_F + 8), b"gamma, beta and zs_p"),
    ("sgrl_layernorm_fwd", dict(zs_p=6), b"gamma, beta and zs_p"),
    ("sgrl_layernorm_fwd", dict(x=_F + 4), b"x and zs_s"),
    ("sgrl_layernorm_fwd", dict(zs_s=2), b"x and zs_s"),
    ("sgrl_layernorm_fwd", dict(T=-1), b"T must be >= 0"),
    ("sgrl_layernorm_bwd", dict(dx=None), b"null pointer"),
    ("sgrl_layernorm_bwd", dict(dbeta=None), b"dgamma and dbeta go together"),
    ("sgrl_layernorm_bwd", dict(rd_y=_F, rd_ldy=128), b"go together"),
    ("sgrl_layernorm_bwd", dict(gamma=_F + 12), b"gamma and zs_p"),
    ("sgrl_layernorm_bwd", dict(nb=17), b"nb must be 1..16"),
    ("sgrl_matapply_fwd", dict(R=None), b"null pointer"),
    ("sgrl_matapply_bwd", dict(dF=None), b"null pointer"),
    ("sgrl_matapply_l5_fwd", dict(Vn=None), b"null pointer"),
    ("sgrl_matapply_l5_bwd", dict(dVn=_F + 4), b"dVn and zs_w"),
    ("sgrl_matapply_l5_bwd", dict(zs_w=2), b"dVn and zs_w"),
    ("sgrl_actor_out_fwd", dict(nb=17), b"nb must be 1..16"),
    ("sgrl_actor_out_bwd", dict(dwd=None), b"null pointer"),
    ("sgrl_rowdiv_bwd", dict(cs_n=769), b"cs_n must be 0..N"),
    ("sgrl_rowdiv_bwd", dict(T=-1), b"T must be >= 0"),
    ("sgrl_colsum", dict(N=0), b"N >= 1"),
    ("sgrl_block_copy", dict(src=None), b"null pointer"),
    ("sgrl_fold_sym", dict(n=18), b"n must be 1..17"),
    ("sgrl_fold_sym", dict(n=0), b"n must be 1..17"),
    ("sgrl_fold_sym", dict(wf=_F + 4), b"fold planes"),
    ("sgrl_fold_sym", dict(plane=1022), b"fold planes"),
    ("sgrl_fold_sym", dict(zs_s=5), b"fold planes"),
    ("sgrl_unfold_sym", dict(rows=None), b"null pointer"),
    ("sgrl_unfold_sym", dict(nb=17), b"nb must be 1..16"),
])
def test_single_kernel_entry_points_refuse_bad_arguments(name, over, msg):
    """Every single-kernel entry point refuses a call its kernel cannot run, before anything is enqueued (fake addresses: a call
    that got as far as a launch would fault, so a refusal is the only way to pass here)."""
    from sgrl_b200 import _lib
    rc = _call(name, **over)
    assert rc < 0 and msg in _lib.lib.sgrl_last_error(), _lib.lib.sgrl_last_error()


def test_single_kernel_entry_points_are_abi_12():
    from sgrl_b200 import _lib
    assert _lib.lib.sgrl_version() == 12
    for name, args in _ARGS.items():
        assert len(getattr(_lib.lib, name).argtypes) == len(args) + 2, name
    # SgrlGemmDesc: four problems and ten int32 fields (n, use_tc, sm2_ok and the seven planner overrides); the library asserts the same size
    assert ctypes.sizeof(_lib.GemmDesc) == 4 * ctypes.sizeof(_lib.GemmProblem) + 40
