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
