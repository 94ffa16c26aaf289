#!/usr/bin/env python
"""K seeds of TD3 on one GPU: one seed-batched update against K single-agent updates, one process.

  python tools/seed_batch_bench.py [--steps 200] [--rounds 2] [--batches 100,256] [--seeds 1,2,4,8] [--sweep]

Workload: 3d_humanoid_9_full at the reference configs' batch sizes (B = 100; B = 256 as in start_humanoid.sh), K seeds each
with its own device batch (synthetic, fixed across steps).  Arms, alternated A/B/A/B:

  A  agents[k].update(batches[k], it) for k = 0..K-1, back to back         K replayed graphs per step
  B  SeedBatchedAgent.update(batches, it)                                  one replayed graph per step

Per arm and round: device ms per step between CUDA events around --steps steps (followed by a synchronise), the ratio
B / A (A is K times the single-agent step), library kernels executed per step (through graph replays and outside them) and
the card's name and power limit, read in the same run.  Prints one JSON line; writes nothing.

--sweep: a hyper-parameter sweep instead of K seeds of one configuration.  Seed k trains with configuration k of
sweep_hparams(K) (learning rate, tau, discount, target-policy noise and gradient clip all differ), in arm B through
SeedBatchedAgent(args, seeds, hparams) and in arm A as an Agent built with those values.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.packed_replay_bench import card  # noqa: E402

MORPH = "3d_humanoid_9_full"


def time_arms(arms, steps, rounds, it, before_window=None):
    """The alternated A/B timing of the seed benchmarks: arms = {name: (fn, agents)}, fn() one step of the arm (reading it[0],
    which is bumped after every step).  Per arm and round: device ms per step between CUDA events around `steps` steps followed
    by a synchronise, wall ms per step on the host clock around the same window (synchronise included), and the library
    kernels executed per step (through graph replays and outside them).  before_window(name), if given, runs untimed before
    each window.  Returns {name: {"device_ms", "wall_ms", "kernels_per_step", "device_ms_median", "wall_ms_median"}}."""
    import time
    import torch
    from sgrl_b200._lib import lib
    res = {k: {"device_ms": [], "wall_ms": [], "kernels_per_step": []} for k in arms}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for name, (fn, ags) in arms.items():
            if before_window is not None:
                before_window(name)
            torch.cuda.synchronize()
            l0 = lib.sgrl_launch_count() + sum(a.graph_replayed_launches for a in ags)
            w0 = time.perf_counter()
            ev0.record()
            for _ in range(steps):
                fn(); it[0] += 1
            ev1.record()
            torch.cuda.synchronize()
            w1 = time.perf_counter()
            r = res[name]
            r["device_ms"].append(round(ev0.elapsed_time(ev1) / steps, 4))
            r["wall_ms"].append(round((w1 - w0) * 1e3 / steps, 4))
            r["kernels_per_step"].append((lib.sgrl_launch_count() + sum(a.graph_replayed_launches for a in ags) - l0) / steps)
    for r in res.values():
        r["device_ms_median"] = statistics.median(r["device_ms"])
        r["wall_ms_median"] = statistics.median(r["wall_ms"])
    return res


def sweep_hparams(K):
    """K distinct configurations around the reference's defaults."""
    return [dict(actor_lr=1e-4 * 2.0 ** (k % 4 - 1), critic_lr=1e-4 * 2.0 ** ((k + 1) % 4 - 1), target_smoothing_tau=0.005 * (1 + k % 3),
                 discount=0.99 - 0.005 * (k % 2), policy_noise=0.1 + 0.05 * (k % 3), noise_clip=0.3 + 0.1 * (k % 3),
                 grad_clipping_value=0.1 * (1 + k % 2)) for k in range(K)]


def run_case(B, K, steps, rounds, warmup, dev, sweep=False):
    import torch
    from sgrl_b200 import graph as G, morphologies as M, synth
    from sgrl_b200.agent import Agent
    from sgrl_b200.config import default_args
    from sgrl_b200.seed_batch import SeedBatchedAgent, args_hparams, args_with
    par = M.ALL[MORPH]
    g = G.build_graph(par, device=dev)
    seeds = list(range(K))
    hps = sweep_hparams(K) if sweep else None
    singles = []
    for s in seeds:
        torch.manual_seed(s)
        if sweep:
            h = {**args_hparams(default_args()), **hps[s]}
            ag = Agent(args_with(default_args(), h))
            ag.actor_optimizer.lr, ag.critic_optimizer.lr = h["actor_lr"], h["critic_lr"]
            singles.append(ag)
        else:
            singles.append(Agent(default_args()))
    sb = SeedBatchedAgent(default_args(), seeds, hparams=hps)
    for ag in singles + [sb]:
        ag.lazy_stats = True
        ag.change_morphology(g)
    batches = [{k: v.to(dev) for k, v in synth.make_batch(B, len(par), seed=100 + s).items()} for s in seeds]
    it = [0]

    def arm_a():
        for ag, b in zip(singles, batches):
            ag.update(b, it[0])

    def arm_b():
        sb.update(batches, it[0])

    arms = {"A_k_agents": (arm_a, singles), "B_seed_batched": (arm_b, [sb])}
    for fn, _ in arms.values():              # eager run + capture of both step kinds
        for _ in range(max(warmup, 4)):
            fn(); it[0] += 1
    torch.cuda.synchronize()
    res = time_arms(arms, steps, rounds, it)
    a, b = res["A_k_agents"]["device_ms_median"], res["B_seed_batched"]["device_ms_median"]
    return {"batch": B, "seeds": K, "sweep": sweep, "limb_tokens_per_seed": B * len(par), "arms": res, "ratio_B_over_A": round(b / a, 4),
            "seed_batched_faster": b < a}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per arm and round (>= 200 for a reported number)")
    ap.add_argument("--rounds", type=int, default=2, help="A/B rounds")
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per arm before the first round (at least 4)")
    ap.add_argument("--batches", default="100,256")
    ap.add_argument("--seeds", default="1,2,4,8")
    ap.add_argument("--sweep", action="store_true", help="seed k trains with configuration k of sweep_hparams(K)")
    a = ap.parse_args()
    Bs = [int(x) for x in a.batches.split(",") if x]
    Ks = [int(x) for x in a.seeds.split(",") if x]
    if a.steps < 1 or a.rounds < 1 or not Bs or not all(1 <= k <= 8 for k in Ks):
        ap.error("--steps and --rounds must be >= 1, --seeds within 1..8")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("seed_batch_bench needs a CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    out = {"metric": "seed_batched_td3_update", "morphology": MORPH, "steps": a.steps, "rounds": a.rounds, **card(0), "cases": []}
    for B in Bs:
        for K in Ks:
            out["cases"].append(run_case(B, K, a.steps, a.rounds, a.warmup, dev, a.sweep))
            torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
