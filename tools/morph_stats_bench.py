#!/usr/bin/env python
"""What the per-morphology statistics of a packed update cost: the same agent stepped with per_morphology off and on, one process.

  python tools/morph_stats_bench.py [--steps 200] [--rounds 2] [--cases 3d_cwhh:100,3d_humanoids:256] [--seeds 4]

Workloads: the "++" training sets the statistics matter most for, at the reference configs' batch sizes: CWHH++ (23
morphologies) at B = 100 and Humanoid++ at B = 256 per morphology.  Every (seed, morphology) has its own device ReplayBuffer
of --rows synthetic rows.  Per case two agents, each timed on its own:

  Agent             update_packed_from_buffers(parts, B, it, per_morphology=...)
  SeedBatchedAgent  update_packed_from_buffers_per_seed(parts_per_seed, B, it, per_morphology=...)   K = --seeds

and per agent four arms, alternated off/on/off_lazy/on_lazy in every round: the flag off and on, with lazy_stats off (every
value a Python float: the reward statistics and, when on, the per-morphology values each cost one device-to-host read per
call) and on (0-dim device tensors, no read).  The arms of one agent share its plan; each arm's graphs are captured before
the first round.  Per arm and round: device ms per step between CUDA events around --steps steps, wall ms per step on the
host clock around the same window (both end in a synchronise), and library kernels executed per step (through graph
replays and outside them: the gather).  The card's name and power limit are read in the same run.  Prints one JSON line;
writes nothing.
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
from tools.seed_packed_bench import make_parts  # noqa: E402

CASES = "3d_cwhh:100,3d_humanoids:256"
ARMS = (("off", False, False), ("on", True, False), ("off_lazy", False, True), ("on_lazy", True, True))


def run_agent(ag, step, steps, rounds, warmup):
    """The four arms of one agent; step(flag, it) is one update."""
    it = [0]

    def arm(flag, lazy):
        def fn():
            ag.lazy_stats = lazy
            step(flag, it[0])
        return fn

    arms = {name: (arm(flag, lazy), [ag]) for name, flag, lazy in ARMS}
    for fn, _ in arms.values():
        for _ in range(max(warmup, 4)):      # eager run + capture of both step kinds, flagged and not
            fn(); it[0] += 1
    res = time_arms(arms, steps, rounds, it)
    for name in ("on", "on_lazy"):
        base = res[name.replace("on", "off")]
        res[name]["device_ratio_to_off"] = round(res[name]["device_ms_median"] / base["device_ms_median"], 4)
        res[name]["wall_ratio_to_off"] = round(res[name]["wall_ms_median"] / base["wall_ms_median"], 4)
    plan = next(iter(ag._plans.values()))
    res["graph_launches"] = {f"actor_step={key[0]} per_morphology={len(key) == 3}": n for key, n in sorted(plan.graph_launches.items())}
    return res


def run_case(name, B, K, steps, rounds, warmup, rows, dev):
    import torch
    from sgrl_b200 import morphologies as M
    from sgrl_b200.agent import Agent
    from sgrl_b200.config import default_args
    from sgrl_b200.seed_batch import SeedBatchedAgent
    names = sorted(M.SETS[name])
    out = {"set": name, "batch": B, "morphologies": len(names), "limb_tokens_per_seed": B * sum(len(M.ALL[n]) for n in names)}
    parts = make_parts(names, 1, rows, dev)[0]
    torch.manual_seed(0)
    ag = Agent(default_args())
    out["agent"] = run_agent(ag, lambda flag, it: ag.update_packed_from_buffers(parts, B, it, per_morphology=flag), steps, rounds, warmup)
    del ag, parts
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    parts_per_seed = make_parts(names, K, rows, dev)
    sb = SeedBatchedAgent(default_args(), list(range(K)))
    out["seed_batched"] = run_agent(sb, lambda flag, it: sb.update_packed_from_buffers_per_seed(parts_per_seed, B, it, per_morphology=flag),
                                    steps, rounds, warmup)
    out["seed_batched"]["seeds"] = K
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per arm and round (>= 200 for a reported number)")
    ap.add_argument("--rounds", type=int, default=2, help="rounds of the four alternated arms")
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per arm before the first round (at least 4)")
    ap.add_argument("--cases", default=CASES, help="comma-separated set:batch pairs")
    ap.add_argument("--seeds", type=int, default=4, help="K of the seed-batched agent (1..8)")
    ap.add_argument("--rows", type=int, default=4096, help="rows per replay buffer")
    a = ap.parse_args()
    cases = [(c.split(":")[0], int(c.split(":")[1])) for c in a.cases.split(",") if c]
    from sgrl_b200 import morphologies as M
    if a.steps < 1 or a.rounds < 1 or not cases or not 1 <= a.seeds <= 8 or any(s not in M.SETS for s, _ in cases):
        ap.error(f"--steps and --rounds must be >= 1, --seeds within 1..8, sets among {sorted(M.SETS)}")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("morph_stats_bench needs a CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    out = {"metric": "per_morphology_stats_cost", "steps": a.steps, "rounds": a.rounds, "rows": a.rows, **card(0), "cases": []}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for name, B in cases:
            out["cases"].append(run_case(name, B, a.seeds, a.steps, a.rounds, a.warmup, a.rows, dev))
            torch.cuda.empty_cache()
            print(json.dumps(out["cases"][-1]), file=sys.stderr, flush=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
