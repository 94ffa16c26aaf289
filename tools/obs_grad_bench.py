#!/usr/bin/env python
"""Cost of asking the backward for d/d(obs): SetNetModule.backward_raw with and without `dobs`, one process.

  python tools/obs_grad_bench.py [--batch 256] [--iters 200] [--rounds 2] [--morph 3d_humanoid_9_full]

Cases: the actor (nb = 1) and the twin critics (nb = 2), full backward with parameter gradients, on one synthetic batch of
--batch graphs of --morph.  Per case, the arms are alternated A/B/A/B (--rounds of each) on the same stash and workspace:

  A  backward_raw(..., dobs=None)            the pass as it was
  B  backward_raw(..., dobs=<(nb,T,41)>)     the same pass plus input_grad_kernel at its end

Per arm and round: device ms per backward between CUDA events around --iters back-to-back calls.  Then a separate
torch.profiler pass (profiler on, so not part of the timings above) gives the device time of input_grad_kernel itself, and
with the algorithmic bytes per token computed from shapes below, its GB/s.  The card's name and power limit are read in
the same run.  Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card(index):
    """Name and power limit of the GPU, read now (nvidia-smi query only)."""
    import torch
    out = {"gpu": torch.cuda.get_device_name(index), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as ex:          # the timing stands without it; say why it is missing
        out["power_limit_w_error"] = repr(ex)
    return out


def bytes_per_token(kind: str, n_layers: int, limbs: int) -> dict:
    """Algorithmic bytes input_grad_kernel moves per token (fp32), from the shapes it reads:
    frame 0 dVg (3x128) and dh (128); the head's dZ1 (3x32, + dZ3 for the actor) and dSH[:17]; per layer the gd columns
    30, 31 of dZ1, dZ2, dZ3 (3 x 3 x 2), the gd channels of d og (3 rows x 2 heads x 2) and the token's column of the
    attention probabilities (2 heads x limbs); the actor's dOut, out and w (3 each).  Written: d obs (41).
    The weight slices staged per CTA (g_encoder 128x8, encoder 128x17, gg_proj / g_proj 30x8) are not per token."""
    actor = kind == "actor"
    r = 3 * 128 + 128 + 96 * (2 if actor else 1) + 17 + n_layers * (18 + 12 + 2 * limbs) + (9 if actor else 0)
    return {"read": 4 * r, "write": 4 * 41, "total": 4 * (r + 41)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--morph", default="3d_humanoid_9_full")
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("obs_grad_bench needs a CUDA device (nothing is timed on the CPU)")
    from oracle import ref_loader
    from sgrl_b200 import graph as G, morphologies as M, synth
    from sgrl_b200.modules import SEPolicy, SECritic

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    args = ref_loader.default_args()
    par = M.ALL[a.morph]
    n = len(par)
    g = G.build_graph(par, device=dev)
    b = synth.make_batch(a.batch, n, seed=1)
    obs = b["obs"].to(dev).view(-1, 41).contiguous()
    act = b["action"].to(dev).view(-1, 3).contiguous()
    result = {"morph": a.morph, "batch": a.batch, "tokens": a.batch * n, "iters": a.iters, **card(0), "cases": {}}

    for kind in ("actor", "critic"):
        torch.manual_seed(0)
        mod = SEPolicy(41, 3, 32, 100, 1.0, None, False, False, False, args) if kind == "actor" else \
            SECritic(41, 3, 32, 100, None, False, False, False, args)
        mod.change_morphology(g)
        nb, od = (1, 3) if kind == "actor" else (2, 1)
        tb = mod._tables(a.batch)
        _, stash = mod.forward_raw(tb, obs, act if kind == "critic" else None, keep=True, nb=nb)
        grads = torch.zeros(mod._nb * mod._live, device=dev)
        ws = torch.empty(mod.ws_floats(tb.T, nb), device=dev)
        dout = torch.randn(nb, tb.T, od, device=dev)
        dobs = torch.empty(nb, tb.T, 41, device=dev)

        def run(with_dobs, iters):
            for _ in range(iters):
                mod.backward_raw(tb, stash, dout, nb, grads, False, trusted_split=True, ws=ws, dobs=dobs if with_dobs else None)

        mod._split_for(tb.T, False)              # the split is fresh from here on: trusted_split keeps it out of the timings
        run(False, a.warmup); run(True, a.warmup)
        torch.cuda.synchronize()
        ms = {"without_dobs": [], "with_dobs": []}
        for _ in range(a.rounds):
            for arm, flag in (("without_dobs", False), ("with_dobs", True)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(flag, a.iters)
                e1.record()
                torch.cuda.synchronize()
                ms[arm].append(e0.elapsed_time(e1) / a.iters)

        # kernel time in a pass of its own (profiler on)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(True, 50)
            torch.cuda.synchronize()
        k_us = [e.device_time_total / e.count for e in prof.key_averages() if "input_grad_kernel" in e.key]
        bpt = bytes_per_token(kind, mod._n_layers, n)
        case = {"nb": nb, "ms_per_backward": {k: [round(x, 4) for x in v] for k, v in ms.items()},
                "delta_ms_median": round(statistics.median(ms["with_dobs"]) - statistics.median(ms["without_dobs"]), 4),
                "bytes_per_token": bpt}
        if k_us:
            t_us = k_us[0]
            case["input_grad_kernel_us"] = round(t_us, 2)
            case["input_grad_kernel_gb_s"] = round(bpt["total"] * tb.T * nb / (t_us * 1e-6) / 1e9, 1)
        result["cases"][kind] = case
    print(json.dumps(result))


if __name__ == "__main__":
    main()
