#!/usr/bin/env python
"""Packed multi-morphology TD3 update fed from per-morphology device replay buffers: two ways, one process.

  python tools/packed_replay_bench.py [--steps 200] [--rounds 2] [--workloads 3d_cwhh,3d_humanoids]

Workloads: 3d_cwhh (23 morphologies, B = 100 each) and 3d_humanoids (6 morphologies, B = 256 each).  Every morphology has a
device ReplayBuffer of 32 768 synthetic rows.  Arms, alternated A/B/A/B on one agent (they share its plan and captured graphs):

  A  agent.update_packed([(g, buf.sample(B)) for g, buf in parts], it)      one index copy + gather per morphology, then
                                                                             five copies per morphology into the plan
  B  agent.update_packed_from_buffers(parts, B, it)                          one index copy, one gather into the plan

Per arm and round: wall-clock ms per step over --steps steps (lazy_stats, one synchronise at the end), device ms per step
between CUDA events recorded at the start and end of the window, and library launches outside the graph per step
(sgrl_launch_count delta).  The card's name and power limit are read in the same run.  Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {"3d_cwhh": 100, "3d_humanoids": 256}
ROWS = 32768


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


def make_parts(names, dev):
    from sgrl_b200 import graph as G, morphologies as M, synth
    from sgrl_b200.buffer import ReplayBuffer
    parts = []
    for i, name in enumerate(names):
        par = M.ALL[name]
        n = len(par)
        buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=ROWS, device=dev)
        b = synth.make_batch(ROWS, n, seed=1000 + i)
        buf.add_batch(*(b[k].to(dev) for k in ("obs", "action", "next_obs", "reward", "done")))
        parts.append((G.build_graph(par, device=dev), buf))
    return parts


def run_workload(set_name, B, steps, rounds, warmup, dev):
    import torch
    from sgrl_b200 import morphologies as M
    from sgrl_b200._lib import lib
    from sgrl_b200.agent import Agent
    from sgrl_b200.config import default_args
    names = sorted(M.SETS[set_name])
    parts = make_parts(names, dev)
    torch.manual_seed(0)
    agent = Agent(default_args())
    agent.lazy_stats = True
    it = [0]

    def arm_a():
        agent.update_packed([(g, buf.sample(B)) for g, buf in parts], it[0])

    def arm_b():
        agent.update_packed_from_buffers(parts, B, it[0])

    arms = {"A_update_packed_of_samples": arm_a, "B_update_packed_from_buffers": arm_b}
    random.seed(0)
    for fn in arms.values():                 # eager run + capture of both step kinds, for each arm's loader
        for _ in range(max(warmup, 4)):
            fn(); it[0] += 1
    torch.cuda.synchronize()
    res = {k: {"wall_ms": [], "device_ms": [], "launches": []} for k in arms}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            l0 = lib.sgrl_launch_count()
            t0 = time.perf_counter()
            ev0.record()
            for _ in range(steps):
                fn(); it[0] += 1
            ev1.record()
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3 / steps
            r = res[name]
            r["wall_ms"].append(round(wall, 4))
            r["device_ms"].append(round(ev0.elapsed_time(ev1) / steps, 4))
            r["launches"].append((lib.sgrl_launch_count() - l0) / steps)
    for r in res.values():
        r["wall_ms_median"] = statistics.median(r["wall_ms"])
        r["device_ms_median"] = statistics.median(r["device_ms"])
    tokens = sum(min(B, buf.max_sample_size) * len(g["parents"]) for g, buf in parts)
    return {"morphologies": len(parts), "batch_per_morphology": B, "limb_tokens_per_step": tokens, "rows_per_buffer": ROWS,
            "plans": len(agent._plans), "arms": res}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per arm and round (>= 200 for a reported number)")
    ap.add_argument("--rounds", type=int, default=2, help="A/B rounds")
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per arm before the first round (at least 4)")
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    a = ap.parse_args()
    names = [w for w in a.workloads.split(",") if w]
    unknown = [w for w in names if w not in WORKLOADS]
    if unknown or a.steps < 1 or a.rounds < 1:
        ap.error(f"unknown workloads {unknown}" if unknown else "--steps and --rounds must be >= 1")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("packed_replay_bench needs a CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    out = {"metric": "packed_update_from_device_buffers", "steps": a.steps, "rounds": a.rounds, **card(0), "workloads": {}}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for w in names:
            out["workloads"][w] = run_workload(w, WORKLOADS[w], a.steps, a.rounds, a.warmup, dev)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
