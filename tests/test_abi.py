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
