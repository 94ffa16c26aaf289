#!/usr/bin/env python
"""K seeds of packed multi-morphology TD3 on one GPU: one seed-batched update against K single-agent updates, one process.

  python tools/seed_packed_bench.py [--steps 200] [--rounds 2] [--cases 3d_hoppers:100,...] [--seeds 1,2,4,8]

Workloads (the "++" training sets at the reference configs' batch sizes): 3d_hoppers, 3d_walkers, 3d_humanoids and 3d_cwhh at
B = 100 per morphology, and 3d_humanoids at B = 256.  Every (seed, morphology) has its own device ReplayBuffer of --rows
synthetic rows.  Arms, alternated A/B/A/B:

  A  agents[k].update_packed_from_buffers(parts[k], B, it) for k = 0..K-1   K index copies, K gathers, K replayed graphs
  B  SeedBatchedAgent.update_packed_from_buffers_per_seed(parts, B, it)    one index copy, one gather, one replayed graph

Per arm and round: device ms per step between CUDA events around --steps steps (followed by a synchronise), the ratio B / A,
library kernels executed per step (through graph replays and outside them), and the peak device memory of one plan (the
growth of torch.cuda.max_memory_allocated over the plan's first steps: one agent's plan for A, the seed-batched plan for B).
Where the K agents' plans and the seed-batched plan do not fit the card together, each arm's window starts by freeing the
other arm's plans and rebuilding its own, untimed (the result says plans_rebuilt_per_window).
The card's name and power limit are read in the same run.  Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.packed_replay_bench import card  # noqa: E402
from tools.seed_batch_bench import time_arms  # noqa: E402

CASES = "3d_hoppers:100,3d_walkers:100,3d_humanoids:100,3d_cwhh:100,3d_humanoids:256"


def make_parts(names, K, rows, dev):
    """parts[k]: seed k's [(graph_dict, ReplayBuffer)] over `names`, every buffer filled with its own synthetic rows."""
    from sgrl_b200 import graph as G, morphologies as M, synth
    from sgrl_b200.buffer import ReplayBuffer
    graphs = [G.build_graph(M.ALL[n], device=dev) for n in names]
    parts = []
    for k in range(K):
        p = []
        for i, (name, g) in enumerate(zip(names, graphs)):
            n = len(M.ALL[name])
            buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=rows, device=dev)
            b = synth.make_batch(rows, n, seed=1000 * k + i)
            buf.add_batch(*(b[x].to(dev) for x in ("obs", "action", "next_obs", "reward", "done")))
            p.append((g, buf))
        parts.append(p)
    return parts


def run_case(name, B, K, steps, rounds, warmup, rows, dev):
    import torch
    from sgrl_b200 import morphologies as M
    from sgrl_b200.agent import Agent
    from sgrl_b200.config import default_args
    from sgrl_b200.seed_batch import SeedBatchedAgent
    names = sorted(M.SETS[name])
    parts = make_parts(names, K, rows, dev)
    singles = []
    for s in range(K):
        torch.manual_seed(s)
        singles.append(Agent(default_args()))
    sb = SeedBatchedAgent(default_args(), list(range(K)))
    for ag in singles + [sb]:
        ag.lazy_stats = True
    it = [0]

    def arm_a():
        for ag, p in zip(singles, parts):
            ag.update_packed_from_buffers(p, B, it[0])

    def arm_b():
        sb.update_packed_from_buffers_per_seed(parts, B, it[0])

    def plan_peak(fn):
        """Device memory the first steps of a fresh plan take at their peak (its buffers, stashes, workspaces, graphs)."""
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        for _ in range(2):                    # eager run + capture of one step kind
            fn(); it[0] += 2
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    peak = {"A_k_agents": plan_peak(lambda: singles[0].update_packed_from_buffers(parts[0], B, it[0])),
            "B_seed_batched": plan_peak(arm_b)}
    arms = {"A_k_agents": (arm_a, singles), "B_seed_batched": (arm_b, [sb])}
    # K agents' plans and the seed-batched plan side by side must fit the card with room to spare; otherwise (CWHH++ at K = 8)
    # each arm's window starts by freeing the other arm's plans and rebuilding its own (eager run + capture, untimed)
    rebuild = K * peak["A_k_agents"] + peak["B_seed_batched"] > 0.8 * torch.cuda.get_device_properties(dev).total_memory

    def warm(fn):
        for _ in range(max(warmup, 4)):      # eager run + capture of both step kinds
            fn(); it[0] += 1

    def before_window(arm):
        """Rebuild mode: free the other arm's plans, then rebuild this arm's (untimed)."""
        fn, ags = arms[arm]
        for other in singles + [sb]:
            if other not in ags:
                other._plans.clear()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        warm(fn)

    if not rebuild:
        for fn, _ in arms.values():
            warm(fn)
    torch.cuda.synchronize()
    res = time_arms(arms, steps, rounds, it, before_window if rebuild else None)
    for k, r in res.items():
        r["plan_peak_bytes"] = peak[k]
    a, b = res["A_k_agents"]["device_ms_median"], res["B_seed_batched"]["device_ms_median"]
    tokens = B * sum(len(M.ALL[n]) for n in names)
    return {"set": name, "batch": B, "morphologies": len(names), "seeds": K, "limb_tokens_per_seed": tokens, "arms": res,
            "plans_rebuilt_per_window": rebuild,
            "ratio_B_over_A": round(b / a, 4), "seed_batched_faster": b < a}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per arm and round (>= 200 for a reported number)")
    ap.add_argument("--rounds", type=int, default=2, help="A/B rounds")
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per arm before the first round (at least 4)")
    ap.add_argument("--cases", default=CASES, help="comma-separated set:batch pairs")
    ap.add_argument("--seeds", default="1,2,4,8")
    ap.add_argument("--rows", type=int, default=4096, help="rows per replay buffer")
    a = ap.parse_args()
    cases = [(c.split(":")[0], int(c.split(":")[1])) for c in a.cases.split(",") if c]
    Ks = [int(x) for x in a.seeds.split(",") if x]
    from sgrl_b200 import morphologies as M
    if a.steps < 1 or a.rounds < 1 or not cases or not all(1 <= k <= 8 for k in Ks) or any(s not in M.SETS for s, _ in cases):
        ap.error(f"--steps and --rounds must be >= 1, --seeds within 1..8, sets among {sorted(M.SETS)}")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("seed_packed_bench needs a CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    out = {"metric": "seed_batched_packed_td3_update", "steps": a.steps, "rounds": a.rounds, "rows": a.rows, **card(0), "cases": []}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for name, B in cases:
            for K in Ks:
                out["cases"].append(run_case(name, B, K, a.steps, a.rounds, a.warmup, a.rows, dev))
                torch.cuda.empty_cache()
                print(json.dumps(out["cases"][-1]), file=sys.stderr, flush=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
