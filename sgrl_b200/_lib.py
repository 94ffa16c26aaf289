"""ctypes binding of libsgrl_b200.so (C ABI declared in include/sgrl_b200.h).

There is no CPU fallback: if the CUDA library is missing the import fails loudly, and every
compute entry point requires CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SGRL_LIB") or os.path.join(_HERE, "libsgrl_b200.so")      # SGRL_LIB: A/B runs of two builds (tools/)

ACTOR, CRITIC = 0, 1


class SgrlError(RuntimeError):
    pass


if not os.path.isfile(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: sgrl_b200 has no CPU/PyTorch fallback. Build the sm_100a library with "
        "`python -c 'import __graft_entry__ as g; g.build()'` or `make -C sgrl_b200/csrc`."
    )

lib = C.CDLL(LIB_PATH)

c_f = C.c_void_p      # device pointers travel as integers
c_i64 = C.c_int64
c_int = C.c_int


class NetCall(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("n_layers", C.c_int32), ("nb", C.c_int32), ("T", C.c_int32),
        ("G", C.c_int32), ("keep", C.c_int32), ("use_tc", C.c_int32), ("max_limbs", C.c_int32),
        ("params", c_f), ("grads", c_f), ("stash", c_f), ("stash_stride", c_i64),
        ("ws", c_f), ("ws_stride", c_i64),
        ("cu_limbs", c_f), ("rel_off", c_f), ("relation", c_f), ("rank3", c_f),
        ("max_action", C.c_float), ("pad_", C.c_float),
        ("params_hi", c_f), ("params_lo", c_f),
    ]


class ReplayPart(C.Structure):
    _fields_ = [
        ("rows", c_f), ("row_floats", c_i64), ("capacity", c_i64),
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("batch", C.c_int32), ("pad_", C.c_int32),
    ]


_PROTOS = {
    "sgrl_version": (c_int, []),
    "sgrl_last_error": (C.c_char_p, []),
    "sgrl_launch_count": (C.c_longlong, []),
    "sgrl_profile": (c_int, [c_int]),
    "sgrl_profile_collect": (c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong), c_int]),
    "sgrl_gemm_trace": (c_int, [c_f]),
    "sgrl_param_count": (c_int, [c_int, c_int]),
    "sgrl_param_info": (c_int, [c_int, c_int, c_int, C.c_char_p, c_int, C.POINTER(c_int), C.POINTER(c_int), C.POINTER(c_i64), C.POINTER(c_int)]),
    "sgrl_arena_floats": (c_int, [c_int, c_int, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "sgrl_stash_floats": (c_i64, [c_int, c_int, c_i64, c_int]),
    "sgrl_ws_floats": (c_i64, [c_int, c_i64]),
    "sgrl_stash_info": (c_int, [c_int, c_int, c_i64, c_int, C.c_char_p, c_int, C.POINTER(c_i64), C.POINTER(c_int)]),
    "sgrl_set_forward": (c_int, [C.POINTER(NetCall), c_f, c_i64, c_f, c_i64, c_f, c_i64, c_f]),
    "sgrl_set_backward": (c_int, [C.POINTER(NetCall), c_f, c_i64, c_int, c_f, c_i64, c_f]),
    "sgrl_inv_feature_fwd": (c_int, [c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_int, c_f]),
    "sgrl_inv_feature_bwd": (c_int, [c_f, c_f, c_f, c_f, c_f, c_int, c_f]),
    "sgrl_attention_fwd": (c_int, [c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_int, c_int, c_f, c_f, c_f, c_f]),
    "sgrl_attention_bwd": (c_int, [c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_int, c_int, c_f, c_f, c_f, c_f]),
    "sgrl_gemm": (c_int, [c_f, c_int, c_int, c_f, c_int, c_int, c_f, c_int, c_int, c_int, c_int, C.c_float, c_f, c_f,
                          c_int, c_int, c_int, c_int, c_f]),
    "sgrl_gemm_presplit": (c_int, [c_f, c_int, c_int, c_f, c_f, c_int, c_int, c_f, c_int, c_int, c_int, c_int, C.c_float, c_f, c_f,
                                   c_int, c_int, c_int, c_f]),
    "sgrl_gemm_gram": (c_int, [c_f, c_f, c_f, c_f, c_f, c_int, c_f, c_f, c_int, c_int, c_int, c_f]),
    "sgrl_gemm_gd": (c_int, [c_f, c_int, c_f, c_f, c_int, c_f, c_f, c_int, c_int, c_f]),
    "sgrl_gemm_pair": (c_int, [c_f, c_int, c_f, c_f, c_f, c_f, c_int, c_int, c_int, c_int, c_f, c_int, c_f, c_f, c_f, c_f, c_int, c_int,
                               c_int, c_int, c_int, c_f]),
    "sgrl_split_tf32": (c_int, [c_f, c_f, c_f, c_i64, c_f]),
    "sgrl_td3_smooth_action": (c_int, [c_f, c_f, c_f, C.c_float, C.c_float, c_i64, c_f]),
    "sgrl_td3_smooth_action_rng": (c_int, [c_f, c_f, c_f, C.c_float, C.c_float, C.c_float, c_i64, C.c_uint64, c_f, c_f]),
    "sgrl_td3_critic_loss": (c_int, [c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, C.c_float, C.c_float, c_int, c_f, c_int, c_f]),
    "sgrl_td3_actor_loss": (c_int, [c_f, c_f, c_f, c_f, c_int, c_f]),
    "sgrl_sumsq": (c_int, [c_f, c_i64, c_f, c_f]),
    "sgrl_adam_clip": (c_int, [c_f, c_f, c_f, c_f, c_i64, c_f, c_f, C.c_double, C.c_double, C.c_double, C.c_double, C.c_float, C.c_float, c_f, c_f, c_f]),
    "sgrl_bump_step": (c_int, [c_f, c_f]),
    "sgrl_polyak": (c_int, [c_f, c_f, c_i64, C.c_float, c_f, c_f, c_i64, c_f]),
    "sgrl_stream_fence": (c_int, [c_f]),
    "sgrl_deterministic": (c_int, [c_int]),
    "sgrl_replay_gather": (c_int, [c_f, c_i64, c_i64, c_f, c_int, c_int, c_int, c_f, c_f, c_f, c_f, c_f, c_f]),
    "sgrl_replay_scatter": (c_int, [c_f, c_i64, c_i64, c_f, c_f, c_int, c_f]),
    "sgrl_replay_gather_packed": (c_int, [C.POINTER(ReplayPart), c_int, c_f, c_f, c_f, c_f, c_f, c_f, c_f]),
}
EXPORTS = tuple(_PROTOS)

for _name, (_res, _args) in _PROTOS.items():
    _fn = getattr(lib, _name)          # AttributeError here = header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise SgrlError(f"{what or 'sgrl call'} failed ({rc}): {lib.sgrl_last_error().decode()}")


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise SgrlError("sgrl_b200 kernels need CUDA tensors; there is no CPU fallback")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


PROF_CLASSES = ("gemm_simt", "gemm_tcgen05", "feature_k1", "attention_k2", "other")


def profile_collect():
    """{class: (ms, work, launches)} since sgrl_profile(1); call after torch.cuda.synchronize()."""
    n = len(PROF_CLASSES)
    ms, work, cnt = (C.c_double * n)(), (C.c_double * n)(), (C.c_longlong * n)()
    check(lib.sgrl_profile_collect(ms, work, cnt, n), "sgrl_profile_collect")
    return {PROF_CLASSES[i]: (ms[i], work[i], cnt[i]) for i in range(n)}


def param_table(kind: int, n_layers: int):
    """[(name, shape, offset, live)] straight from the library (single source of truth)."""
    n = lib.sgrl_param_count(kind, n_layers)
    if n <= 0:
        raise SgrlError(lib.sgrl_last_error().decode())
    out = []
    buf = C.create_string_buffer(192)
    rows, cols, live, off = c_int(), c_int(), c_int(), c_i64()
    for i in range(n):
        check(lib.sgrl_param_info(kind, n_layers, i, buf, 192, C.byref(rows), C.byref(cols), C.byref(off), C.byref(live)))
        shape = (rows.value, cols.value) if cols.value else (rows.value,)
        out.append((buf.value.decode(), shape, off.value, bool(live.value)))
    return out


def arena_floats(kind: int, n_layers: int):
    a, b = c_i64(), c_i64()
    check(lib.sgrl_arena_floats(kind, n_layers, C.byref(a), C.byref(b)))
    return a.value, b.value


def stash_info(kind, n_layers, T, keep, name, layer=-1):
    off, per = c_i64(), c_int()
    check(lib.sgrl_stash_info(kind, n_layers, T, keep, name.encode(), layer, C.byref(off), C.byref(per)))
    return off.value, per.value
