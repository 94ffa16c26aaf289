"""K1, the invariant features, through the C ABI (sgrl_inv_feature_fwd / sgrl_inv_feature_bwd) against the fp64
references of tests/kernel_ref.py, in every launch regime:

  inv_feature_small_fwd_kernel   T <= 128: one warp per token
  inv_feature_fwd_kernel         T > 128: 32-token tiles (a partial last tile when T % 32 != 0), CTAs walking several tiles
                                 above 4 CTAs/SM x 148 tiles (~19 K tokens)
  inv_feature_bwd_kernel         one warp per token, at most 8 x 148 CTAs of 8 warps: warps walk tokens above 9 472

Per-token errors, NaN-prefilled outputs with pad rows past T, the 16 padding slots of the packed Gram exactly 0, and the
kernel that ran asserted from a torch.profiler trace (taken in a separate process)."""
import pytest
import torch

import kernel_ref as R
from sgrl_b200.packing import pack_indices

pytestmark = pytest.mark.gpu

PAD = 3
SLOTS = pack_indices()[0]
PAD_SLOTS = sorted(set(range(544)) - set(SLOTS))


def token_err(got, ref):
    """worst per-token relative error and its token."""
    T = ref.shape[0]
    got, ref = got.double().reshape(T, -1), ref.reshape(T, -1)
    e = (got - ref).norm(dim=1) / ref.norm(dim=1).clamp_min(1e-300)
    t = int(e.argmax())
    return e[t].item(), t


def sentinel(T, *shape):
    return torch.full((T + PAD, *shape), float("nan"), device="cuda")


FWD_T = [1, 7, 128, 129, 2304, 2305, 20001]

# Kernel names of every forward case, traced with torch.profiler in a process of their own: inside a long pytest process
# the trace of these launches has been seen to come back with the runtime call but without the kernel's activity record.
_TRACE = r"""
import json, torch
from torch.profiler import ProfilerActivity, profile
from sgrl_b200._lib import lib, ptr, stream, check
out = {}
for T in %s:
    for head in (0, 1):
        for nproj in (1, 2):
            C = 136 if head else 128
            e = lambda *s: torch.zeros(*s, device="cuda")
            X, v0, gd, P1 = e(T, 3, 128), e(T, 3, 8) if head else None, e(T, 3, 2), e(30, C)
            P2, Z2 = (e(30, C), e(T, 3, 32)) if nproj == 2 else (None, None)
            Z, G, F = e(T, 3, 32), e(T, 544), e(T)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                check(lib.sgrl_inv_feature_fwd(ptr(X), ptr(v0), ptr(gd), ptr(P1), ptr(P2), ptr(Z), ptr(Z2), ptr(G), ptr(F), T, stream()))
                torch.cuda.synchronize()
            out["%%d,%%d,%%d" %% (T, head, nproj)] = [ev.name for ev in prof.events() if "inv_feature" in ev.name]
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def traced_kernels():
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _TRACE % (FWD_T,)], cwd=root, capture_output=True, text=True,
                       env=dict(os.environ, PYTHONPATH=os.pathsep.join([root, os.environ.get("PYTHONPATH", "")])))
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("nproj", [1, 2])
@pytest.mark.parametrize("head", [False, True], ids=["C128", "C136"])
@pytest.mark.parametrize("T", FWD_T)
def test_inv_feature_forward(traced_kernels, T, head, nproj):
    from sgrl_b200._lib import lib, ptr, stream, check
    g = torch.Generator(device="cuda").manual_seed(T * 4 + head * 2 + nproj)
    C = 136 if head else 128
    X = torch.randn(T, 3, 128, device="cuda", generator=g)
    v0 = torch.randn(T, 3, 8, device="cuda", generator=g) if head else None
    gd = torch.randn(T, 3, 2, device="cuda", generator=g)
    P1 = torch.randn(30, C, device="cuda", generator=g) / C ** 0.5
    P2 = torch.randn(30, C, device="cuda", generator=g) / C ** 0.5 if nproj == 2 else None
    Z, G, F = sentinel(T, 3, 32), sentinel(T, 544), sentinel(T)
    Z2 = sentinel(T, 3, 32) if nproj == 2 else None
    check(lib.sgrl_inv_feature_fwd(ptr(X), ptr(v0), ptr(gd), ptr(P1), ptr(P2), ptr(Z), ptr(Z2), ptr(G), ptr(F), T, stream()),
          "sgrl_inv_feature_fwd")
    torch.cuda.synchronize()
    want = "inv_feature_small_fwd_kernel" if T <= 128 else "inv_feature_fwd_kernel"
    names = traced_kernels[f"{T},{int(head)},{nproj}"]
    assert names and all(want in n for n in names), f"expected {want}, the trace shows {names}"

    outs = (Z, G, F) + ((Z2,) if nproj == 2 else ())
    for buf in outs:
        assert torch.isnan(buf[T:]).all(), "a pad row past T was written"
        assert torch.isfinite(buf[:T]).all(), "a row < T was left unwritten or is not finite"
    assert torch.all(G[:T, PAD_SLOTS] == 0.0), "the padding slots of the packed Gram must be written as 0"
    rZ, rZ2, rG, rF = R.inv_feature_fwd_ref(X, v0, gd, P1, P2)
    for name, got, ref in (("Z", Z[:T], rZ), ("G", G[:T], rG), ("F", F[:T, None], rF[:, None])) + \
                          ((("Z2", Z2[:T], rZ2),) if nproj == 2 else ()):
        e, t = token_err(got, ref)
        assert e <= 1e-6, f"{name}: token {t} of {T} rel err {e:.2e}"
    assert torch.equal(Z[:T, :, 30:], gd) and (nproj == 1 or torch.equal(Z2[:T, :, 30:], gd))


@pytest.mark.parametrize("T", [1, 9473])
def test_inv_feature_backward(T):
    """dZ on all 32 columns (the state gradient uses the gd columns 30, 31) at <= 1e-5 per token; NaN in the padding slots
    of dGp must not reach dZ; a token with Z = 0 (F - 1 = ||G|| = 0) gets dZ = 0, not NaN."""
    from sgrl_b200._lib import lib, ptr, stream, check
    g = torch.Generator(device="cuda").manual_seed(T)
    Z = torch.randn(T, 3, 32, device="cuda", generator=g)
    zero = T // 2 if T > 1 else None
    if zero is not None:
        Z[zero] = 0.0
    Gfull, _ = R.gram_packed(Z.double())
    F = (torch.linalg.matrix_norm(Gfull) + 1.0).float()
    dG = torch.randn(T, 544, device="cuda", generator=g)
    dG[:, PAD_SLOTS] = float("nan")
    dF = torch.randn(T, device="cuda", generator=g) * 0.1
    dZ = sentinel(T, 3, 32)
    check(lib.sgrl_inv_feature_bwd(ptr(dG), ptr(dF), ptr(Z), ptr(F), ptr(dZ), T, stream()), "sgrl_inv_feature_bwd")
    torch.cuda.synchronize()
    assert torch.isnan(dZ[T:]).all(), "a pad row past T was written"
    assert torch.isfinite(dZ[:T]).all(), "a row < T was left unwritten or is not finite (NaN from the padding slots?)"
    keep = torch.ones(T, dtype=torch.bool, device="cuda")
    if zero is not None:
        assert torch.all(dZ[zero] == 0.0)
        keep[zero] = False
    ref = R.inv_feature_bwd_ref(dG, dF, Z)
    e, t = token_err(dZ[:T][keep], ref[keep])
    assert e <= 1e-5, f"dZ: token {t} rel err {e:.2e}"
