#!/usr/bin/env python
"""Benchmark of the SET TD3 hot path (BASELINE.json: "SET TD3 update samples/sec and rollout
limb-tokens/sec at 1/2/4/8 B200").

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels via the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU

A "step" is one `Agent.update` (TD3 update, src/agent.py:117-183) on one synthetic replay
minibatch of the named morphology (default: 3d_humanoid_9_full, N=9 limbs, B=256 — the batch
start_humanoid.sh really samples, src/configs/default.py:61); even `it` includes the delayed
actor step + Polyak.  --steps K timed steps run, exactly K, each from the same seeded initial
state (restored outside the timed window).  N>1: one process per GPU (torchrun),
every rank draws its own minibatch (weak scaling) and the flat gradient arena is all-reduced
over NCCL before the fused clip+Adam pass.  One JSON line is printed by rank 0.

--dump-outputs DIR writes what the last timed step returned and the parameters it left behind as
DIR/<name>.npy (rank 0).  Inputs and initial weights are seeded, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_TOKEN_UPDATE = 115.1e6      # SURVEY.md §8d / BASELINE.md §3 (reference-executed work, policy_freq=2 average)
FLOP_PER_TOKEN_ACTOR_FWD = 10.14e6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--morph", default="3d_humanoid_9_full")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rollout-envs", type=int, default=16384)
    ap.add_argument("--use-tc", type=int, default=-1, help="1: tcgen05 3xTF32 projections, 0: fp32 SIMT, -1: library default")
    ap.add_argument("--set", default="", help="morphology set (3d_hoppers, 3d_walkers, 3d_humanoids, 3d_cheetahs, 3d_cwhh): one step = one "
                    "update of EVERY morphology of the set at --batch samples each (sharded round-robin over the ranks)")
    ap.add_argument("--packed", action="store_true", help="with --set: all morphologies of the rank in ONE packed update (Agent.update_packed) "
                    "instead of the reference's one-after-the-other schedule (src/trainer.py:245-250)")
    ap.add_argument("--check-replicas", action="store_true", help="after the run, compare the parameter arenas of all ranks bit for bit")
    ap.add_argument("--rollout-sweep", default="", help="comma-separated env counts per GPU (BASELINE config 5: 1K-64K parallel humanoid envs): "
                    "adds rollout_sweep = [{envs_per_gpu, ms_per_forward, value}, ...] to the line, same timing as the rollout leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-rollout", action="store_true")
    ap.add_argument("--no-bf16", action="store_true", help="skip the separately reported BF16-input leg")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the last timed step's loss dict and a fixed sample of the "
                    "updated parameters as DIR/<name>.npy; with --set and without --packed, every morphology's loss dict, its "
                    "name as prefix (<morphology>_loss_critic_loss.npy, ...)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "src": "fallback"}


DUMP_SAMPLE = 1 << 21      # parameters kept per network in a dump: 4 nets x 8 MB, under the 64 MB a dump may take


def dump_outputs(path, ld, agent):
    """What a caller of the timed path holds after its last step: the loss dict Agent.update returned (one .npy per key, '/'
    -> '_', float64) and the parameters of the four networks (<net>_params.npy, float32).  An arena larger than DUMP_SAMPLE
    floats is sampled at positions drawn from a fixed seed, the same positions in every run."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for k, v in ld.items():
        np.save(os.path.join(path, k.replace("/", "_") + ".npy"), torch.as_tensor(v).detach().double().cpu().reshape(-1).numpy())
    for name in ("actor", "critic", "actor_target", "critic_target"):
        flat = getattr(agent, name).full_arena.detach()
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(1234))[:DUMP_SAMPLE].sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(path, name + "_params.npy"), flat.float().cpu().numpy())


def snapshot(agent):
    """Copies of the state an update carries to the next one: the four networks' arenas and both optimizers' moments and
    step counts."""
    opts = (agent.actor_optimizer, agent.critic_optimizer)
    return ([m.full_arena.detach().clone() for m in (agent.actor, agent.actor_target, agent.critic, agent.critic_target)],
            [t.clone() for o in opts for t in (o.exp_avg, o.exp_avg_sq, o.step_count)])


def restore(agent, snap):
    """Write a snapshot back in place (the captured graphs keep their pointers) and re-derive the tf32 split of every
    network that has one, so that the next update finds it fresh and launches nothing extra."""
    import torch
    nets, state = snap
    opts = (agent.actor_optimizer, agent.critic_optimizer)
    with torch.no_grad():
        for m, x in zip((agent.actor, agent.actor_target, agent.critic, agent.critic_target), nets):
            m.full_arena.copy_(x)
            if m._split is not None:
                m.refresh_split()
        for t, x in zip([t for o in opts for t in (o.exp_avg, o.exp_avg_sq, o.step_count)], state):
            t.copy_(x)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------
def _cpu_steppers(morph, batch):
    """(kind, step(it)) callables for one TD3 update on this host's cores: the LIVE reference (src/agent.py Agent.update,
    unmodified, imported by oracle/ref_loader from /root/reference/src, baseline/_ref/src or $SGRL_REF) when it is on this
    machine, and always the oracle port (oracle/set_oracle.TD3Oracle)."""
    import torch
    from oracle import ref_loader, set_oracle as O
    from sgrl_b200 import graph as G, morphologies as M, synth
    par = M.ALL[morph]
    pa = {"actor." + k: v for k, v in O.synth_params("actor", 11).items()}
    pc = {"critic1." + k: v for k, v in O.synth_params("critic", 12).items()}
    pc.update({"critic2." + k: v for k, v in O.synth_params("critic", 13).items()})
    b = synth.make_batch(batch, len(par), seed=1)
    out = {}
    if ref_loader.find_reference():
        try:
            import contextlib
            with contextlib.redirect_stdout(sys.stderr):      # the reference prints its argument sizes: keep stdout to the JSON line
                ref = ref_loader.load_reference()
                g = ref.utils.getGraphDict(par, ["pre", "inlcrs", "postlcrs"], device=torch.device("cpu"))
                ag = ref.agent.Agent(ref_loader.default_args())
            sd = {}
            for pre in ("actor.", "actor_target."):
                sd.update({pre + k: v.clone() for k, v in pa.items()})
            for pre in ("critic.", "critic_target."):
                sd.update({pre + k: v.clone() for k, v in pc.items()})
            ag.load_state_dict(sd)
            ag.change_morphology(g)
            out["reference"] = lambda it: ag.update(b, it)
        except Exception as ex:      # missing host-only dependency of the reference tree: say so, fall back to the port
            sys.stderr.write(f"bench: live reference not usable ({type(ex).__name__}: {ex}); timing the oracle port\n")
    g2 = G.build_graph(par)
    td3 = O.TD3Oracle(pa, pc)
    noise = torch.randn(batch, 3 * len(par)) * 0.2
    out["port"] = lambda it: td3.update(b, it, noise, g2)
    return out


def cpu_reference_rate(morph, batch, budget_s=20.0, steps=None, warmup=1, threads=None):
    """The reference's CPU implementation of Agent.update timed on this host's cores: the live reference when present
    (kind "reference"), else the oracle port (kind "port": torch CPU ops + torch Adam + clip_grad_norm_, the same math).
    When both exist the port is timed on two updates as well and the port/reference time ratio is reported."""
    import torch
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    steppers = _cpu_steppers(morph, batch)
    kind = "reference" if "reference" in steppers else "port"
    step = steppers[kind]
    it = 0
    for _ in range(max(warmup, 1)):
        t0 = time.perf_counter(); step(it); it += 1
        one = time.perf_counter() - t0
    if steps is None:
        steps = max(2, int(budget_s / max(one, 1e-3)) // 2 * 2)
        steps = min(steps, 20)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(it); it += 1
    dt = time.perf_counter() - t0
    r = {"value": batch * steps / dt, "unit": "samples/s", "cores": threads, "kind": kind,
         "sample": f"{steps} TD3 updates (policy_freq=2) of {morph} B={batch} with " +
                   ("the unmodified reference Agent.update (src/agent.py:117-183)" if kind == "reference" else
                    "the oracle port of src/agent.py:117-183") + f" on {threads} host threads, {dt:.1f}s",
         "ms_per_update": 1e3 * dt / steps}
    if kind == "reference":
        port = steppers["port"]
        port(0); port(1)
        t0 = time.perf_counter(); port(2); port(3)
        r["port_over_reference_time"] = (time.perf_counter() - t0) / 2 / (dt / steps)
    return r


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = a.steps
    # bound the sample so the whole run ends within a few minutes: shrink the per-step batch if needed
    probe = cpu_reference_rate(a.morph, a.batch, steps=2, warmup=1)
    batch = a.batch
    est = probe["ms_per_update"] * 1e-3 * (steps + a.warmup)
    while est > 240 and batch > 16:
        batch //= 2; est /= 2
    r = cpu_reference_rate(a.morph, batch, steps=steps, warmup=max(a.warmup, 1))
    from sgrl_b200 import morphologies as M
    line = {"impl": "reference", "metric": "SET TD3 update samples/sec", "value": r["value"], "unit": "samples/s", "n_gpus": a.gpus,
            "steps": steps, "warmup": a.warmup, "ms_per_step": r["ms_per_update"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{a.morph} TD3 Agent.update, B={a.batch}, N={len(M.ALL[a.morph])} limbs, policy_freq=2", "cpu_sample_batch": batch},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "port_over_reference_time") if k in r},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------
def run_ours(a):
    import torch
    import torch.distributed as dist
    from sgrl_b200 import _lib, graph as G, morphologies as M, synth
    from sgrl_b200.agent import Agent
    from sgrl_b200.config import default_args

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = a.steps, a.warmup              # exactly as asked (the contract wants W >= 3: the default is 6)
    par = M.ALL[a.morph]
    N, B = len(par), a.batch
    torch.manual_seed(0)
    agent = Agent(default_args())
    if a.use_tc >= 0:
        for m in (agent.actor, agent.actor_target, agent.critic, agent.critic_target):
            m.use_tc = a.use_tc
    use_tc = int(agent.actor.use_tc)
    if world > 1:                                   # identical replicas: broadcast rank 0's weights
        for m in (agent.actor, agent.actor_target, agent.critic, agent.critic_target):
            dist.broadcast(m.full_arena, 0)
    g = G.build_graph(par, device=dev)
    agent.change_morphology(g)
    # every timed step starts from this seeded state (restored outside the timed window): fp32 atomics make updates differ
    # from run to run in the last bits, and a trajectory of updates grows that into ~1e-4 (Adam turns the sign of a ~0
    # gradient into a full step), while one update from a fixed state reproduces to rounding
    init = snapshot(agent)
    if a.set:
        return run_set(a, agent, dev, world, rank, local, init)
    nbat = 8
    host = [synth.make_batch(B, N, seed=100 + 17 * rank + i) for i in range(nbat)]
    host = [{k: v.pin_memory() for k, v in b.items()} for b in host]
    devb = [{k: v.to(dev) for k, v in b.items()} for b in host]
    noise = [torch.randn(B, 3 * N, device=dev) * 0.2 for _ in range(nbat)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    agent.lazy_stats = True
    # set-up (not warm-up): the first two updates of a plan run eagerly (one per kind of step), the next two are captured as
    # CUDA graphs; from here on every update is a replay.  `it` keeps counting so actor steps alternate through all phases.
    it = 0
    for _ in range(4):
        agent.update(devb[it % nbat], it, noise=noise[it % nbat]); it += 1
    for _ in range(W):
        agent.update(devb[it % nbat], it, noise=noise[it % nbat]); it += 1
    barrier()
    # ---- timed: K updates, inputs resident in HBM, L2 flushed between steps (outside the event pairs)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = _lib.lib.sgrl_launch_count() + agent.graph_replayed_launches
    barrier()
    for i in range(K):
        r0 = _lib.lib.sgrl_launch_count()
        restore(agent, init)
        l0 += _lib.lib.sgrl_launch_count() - r0          # the split refresh of the restore is not part of the step
        flush.zero_()
        ev[i][0].record()
        ld = agent.update(devb[it % nbat], it, noise=noise[it % nbat]); it += 1
        ev[i][1].record()
    barrier()
    launches = (_lib.lib.sgrl_launch_count() + agent.graph_replayed_launches - l0) / K
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, ld, agent)
    total_ms = sum(s.elapsed_time(e) for s, e in ev)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    value = world * B * K / (total_ms * 1e-3)

    # ---- e2e: the public call with HOST (pinned) buffers, result read back every step
    agent.lazy_stats = False
    for _ in range(4 + min(W, 4)):      # host batches draw the target-policy noise in the kernel: their own pair of graphs (2 eager runs + 2 captures)
        agent.update(host[it % nbat], it)["loss/critic_loss"].item(); it += 1
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        ld = agent.update(host[it % nbat], it); it += 1
        ld["loss/critic_loss"].item()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = world * B * K / t.item()
    h2d = sum(v.numel() * 4 for v in host[0].values())

    line = {"metric": "SET TD3 update samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (3xTF32 tensor-core projections, fp32 accumulate)" if use_tc else "f32", "data": "synthetic",
            "config": {"workload": f"{a.morph} TD3 Agent.update, B={B} per GPU, N={N} limbs, policy_freq=2 (Humanoid++ of start_humanoid.sh)",
                       "l2": "256 MiB buffer written between timed steps (L2 flushed); working set (4 nets + Adam state + grads ~ 300 MB) exceeds L2 anyway",
                       "use_tc": use_tc, "updates_per_s": world * K / (total_ms * 1e-3), "limb_tokens_per_s": value * N},
            "e2e": {"value": e2e_val, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "how": "Agent.update(batch of pinned host tensors, it) + critic_loss.item(), wall clock, max over ranks"},
            "gpu_launches": launches}
    if rank == 0:
        line["clocks"] = clk

    # ---- roofline pass: device time per kernel class (CUDA events on the launching stream), 2 updates
    pk = peaks()
    barrier()
    graphs_on = agent.use_graphs
    agent.use_graphs = False          # the per-class timing pass brackets single launches with events: eager, one stream
    _lib.lib.sgrl_profile(1)
    for i in range(2):
        agent.update(devb[i % nbat], i, noise=noise[i % nbat])
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.lib.sgrl_profile(0)
    agent.use_graphs = graphs_on
    step_ms = total_ms / K
    ser_ms = max(sum(v[0] for v in prof.values()), 1e-9)     # the timing pass runs the launches one by one (no overlap)
    classes = {}
    for name, (ms, work, cnt) in prof.items():
        if cnt:
            classes[name] = {"ms_per_step": ms / 2, "launches_per_step": cnt / 2, "share_of_serialized": ms / ser_ms}
            if name.startswith("gemm"):
                classes[name]["tflops"] = work / (ms * 1e-3) / 1e12
            else:
                classes[name]["gbs"] = work / (ms * 1e-3) / 1e9
    dom = max(classes, key=lambda k: classes[k]["ms_per_step"]) if classes else None
    if dom and dom.startswith("gemm"):
        # algorithmic FLOPs of one update (SURVEY.md 8d: 115.1 MFLOP per limb-token as the reference executes it; >= 98 % of them
        # are the projections) / summed device time of the class in one update.  The kernel EXECUTES fewer (the symmetric Gram is
        # contracted as its triangle: K = 544 instead of 1024) and each costs 3 tf32 MMAs (3xTF32 for fp32 parity), so against the
        # bf16 peak the ceiling of `frac` for this kernel is 1/6.
        alg = FLOP_PER_TOKEN_UPDATE * B * N
        ach = alg / (classes[dom]["ms_per_step"] * 1e-3) / 1e12
        line["roofline"] = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                            "frac": ach / pk["tflops_sustained"], "traffic": 5.84e6, "traffic_unit": "bytes of DRAM traffic per launch",
                            "traffic_src": "mean of 12 launches of this class on the final tree, ncu --set full (profiles/r05u_ncu_gemm_update_summary.txt; "
                                           "r03c_* mid-round: 6.73 MB): 5.84 MB read + 0 MB written (ncu flushes the caches before each launch; in the "
                                           "step the activations and weights of a B=256 update stay in the 126 MB L2)",
                            "peak_src": pk["src"] + " bf16 sustained",
                            "algorithmic_flops_per_step": alg, "launches_per_step": classes[dom]["launches_per_step"],
                            "executed_tflops": classes[dom]["tflops"], "ceiling_frac_3xtf32": 1.0 / 6.0,
                            "frac_of_3xtf32_ceiling": 6.0 * ach / pk["tflops_sustained"],
                            "whole_step_tflops": alg / (step_ms * 1e-3) / 1e12,
                            "note": "B=256 x 9 limbs = 2304 rows per projection: 18 row tiles, launch/latency bound (profiles/r01l_phase_probe.txt); "
                                    "the same kernel at rollout size is reported under rollout.gemm_*"}
    elif dom:
        ach = classes[dom]["gbs"]
        line["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                            "traffic": None, "peak_src": pk["src"]}
    line["kernel_classes"] = classes

    # ---- rollout: SEPolicy.forward under no_grad over many parallel envs (inputs resident)
    if not a.no_rollout:
        E = a.rollout_envs
        obs = synth.make_obs(min(E, 4096), N, seed=7).to(dev)
        obs = obs.repeat((E + obs.shape[0] - 1) // obs.shape[0], 1)[:E].contiguous()
        with torch.no_grad():
            for _ in range(3):
                agent.actor(obs)
            barrier()
            R = 10
            evr = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(R)]
            for i in range(R):
                flush.zero_()
                evr[i][0].record(); agent.actor(obs); evr[i][1].record()
            barrier()
            ms = sum(s.elapsed_time(e) for s, e in evr)
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            tok = world * E * N * R / (t.item() * 1e-3)
            _lib.lib.sgrl_profile(1)
            agent.actor(obs)
            torch.cuda.synchronize()
            rp = _lib.profile_collect()
            _lib.lib.sgrl_profile(0)
        line["rollout"] = {"value": tok, "unit": "limb-tokens/s", "envs_per_gpu": E, "ms_per_forward": t.item() / R,
                           "tflops": tok * FLOP_PER_TOKEN_ACTOR_FWD / 1e12,
                           "feature_k1_gbs": rp["feature_k1"][1] / max(rp["feature_k1"][0], 1e-9) / 1e6,
                           "attention_k2_gbs": rp["attention_k2"][1] / max(rp["attention_k2"][0], 1e-9) / 1e6,
                           "gemm_tflops": (rp["gemm_simt"][1] + rp["gemm_tcgen05"][1]) / max(rp["gemm_simt"][0] + rp["gemm_tcgen05"][0], 1e-9) / 1e9,
                           "gemm_frac_of_3xtf32_ceiling": 6.0 * (rp["gemm_simt"][1] + rp["gemm_tcgen05"][1]) / max(rp["gemm_simt"][0] + rp["gemm_tcgen05"][0], 1e-9) / 1e9 / pk["tflops_sustained"],
                           "hbm_peak_gbs": pk["hbm_gbs"],
                           "feature_k1_frac": rp["feature_k1"][1] / max(rp["feature_k1"][0], 1e-9) / 1e6 / pk["hbm_gbs"],
                           "attention_k2_frac": rp["attention_k2"][1] / max(rp["attention_k2"][0], 1e-9) / 1e6 / pk["hbm_gbs"],
                           "share_ms": {k: v[0] for k, v in rp.items()},
                           "traffic_ncu": {"feature_k1": {"dram_bytes_per_launch": 550.5e6, "algorithmic_bytes_per_launch": 4124.0 * 147456,
                                                          "src": "profiles/r01k_ncu_k1_k2_summary.txt (T=147456)"}}}

    if a.rollout_sweep:
        sweep = []
        for E in [int(x) for x in a.rollout_sweep.split(",") if x]:
            obs = synth.make_obs(min(E, 4096), N, seed=7).to(dev)
            obs = obs.repeat((E + obs.shape[0] - 1) // obs.shape[0], 1)[:E].contiguous()
            with torch.no_grad():
                for _ in range(3):
                    agent.actor(obs)
                barrier()
                R = 10
                evr = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(R)]
                for i in range(R):
                    flush.zero_()
                    evr[i][0].record(); agent.actor(obs); evr[i][1].record()
                barrier()
                t = torch.tensor([sum(s.elapsed_time(e) for s, e in evr)], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sweep.append({"envs_per_gpu": E, "limb_tokens_per_gpu": E * N, "ms_per_forward": t.item() / R,
                          "value": world * E * N * R / (t.item() * 1e-3), "unit": "limb-tokens/s (all GPUs)"})
            del obs
            torch.cuda.empty_cache()
        line["rollout_sweep"] = sweep

    # ---- callers either side of the path (SURVEY.md 8f rank 2 and 4), rank-local, wall clock through the public calls
    if not a.no_rollout:
        import random
        from sgrl_b200.buffer import ReplayBuffer
        cap = 32768
        rb = ReplayBuffer(41 * N, 3 * N, max_buffer_size=cap, device=dev)
        fill = synth.make_batch(cap, N, seed=5)
        rb.add_batch(*(fill[k].to(dev) for k in ("obs", "action", "next_obs", "reward", "done")))
        random.seed(rank)
        agent.lazy_stats = True
        for i in range(4):
            agent.update_from_buffer(rb, B, i)
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            ld = agent.update_from_buffer(rb, B, i)
        ld["loss/critic_loss"].item()
        barrier()
        dt_rb = time.perf_counter() - t0
        evg = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        idx = torch.randint(0, cap, (4096,), device=dev)
        outs = [torch.empty(4096, w, device=dev) for w in (41 * N, 3 * N, 41 * N, 1, 1)]
        rb.gather_into(idx, *outs)
        evg[0].record()
        for _ in range(20):
            rb.gather_into(idx, *outs)
        evg[1].record(); torch.cuda.synchronize()
        line["replay"] = {"value": world * B * K / dt_rb, "unit": "samples/s", "how": "Agent.update_from_buffer(device-resident ReplayBuffer, B, it): "
                          "host draws B indices (random.sample), one gather kernel fills the update graph's inputs; wall clock",
                          "h2d_bytes_per_step": 8 * B, "gather_gbs_B4096": 20 * 4096 * 8.0 * rb.row_floats / (evg[0].elapsed_time(evg[1]) * 1e-3) / 1e9}
        agent.lazy_stats = False
        # acting: B=1 select_action (the reference's per-env call) and the batched front-end over a mixed set of envs
        one = synth.make_obs(1, N, seed=3)[0].numpy().astype("float64")
        for _ in range(5):
            agent.select_action(one)
        t0 = time.perf_counter()
        for _ in range(200):
            agent.select_action(one)
        us_one = (time.perf_counter() - t0) / 200 * 1e6
        names = sorted(M.SETS["3d_humanoids"]) * 4
        gl = {n: G.build_graph(M.SETS["3d_humanoids"][n], device=dev) for n in set(names)}
        ol = [synth.make_obs(1, len(M.SETS["3d_humanoids"][n]), seed=i)[0].numpy() for i, n in enumerate(names)]
        gs = [gl[n] for n in names]
        for _ in range(5):
            agent.select_actions(ol, gs)
        t0 = time.perf_counter()
        for _ in range(100):
            agent.select_actions(ol, gs)
        us_all = (time.perf_counter() - t0) / 100 * 1e6
        agent.change_morphology(g)
        line["acting"] = {"select_action_us": us_one, "select_actions_us": us_all, "envs": len(names),
                          "us_per_env_batched": us_all / len(names),
                          "how": "numpy obs in, numpy actions out (pinned H2D + replayed CUDA graph + D2H + sync); batched = one packed "
                                 "forward over %d Humanoid++ envs of 6 morphologies (src/trainer.py:174-196 does them one by one)" % len(names)}

    # ---- BF16-input mode, stated separately (north_star): the same update / rollout with use_tc = 2 — both operands of every
    # tcgen05 projection rounded to bf16, ONE MMA pass, fp32 accumulate (tests/test_bf16_mode_gpu.py records its accuracy:
    # 1e-3..1e-2 against the oracle, i.e. outside the parity bar).  Never the headline value.
    if not a.no_bf16 and use_tc:
        mods = (agent.actor, agent.actor_target, agent.critic, agent.critic_target)
        for m in mods:
            m.use_tc = 2
        agent.lazy_stats = True
        for _ in range(8):
            agent.update(devb[it % nbat], it, noise=noise[it % nbat]); it += 1
        barrier()
        Kb = min(K, 40)
        evb = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Kb)]
        for i in range(Kb):
            flush.zero_()
            evb[i][0].record()
            agent.update(devb[it % nbat], it, noise=noise[it % nbat]); it += 1
            evb[i][1].record()
        barrier()
        t = torch.tensor([sum(s.elapsed_time(e) for s, e in evb)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        bfl = {"dtype": "bf16 inputs / f32 accumulate, one tcgen05 pass (use_tc=2)", "value": world * B * Kb / (t.item() * 1e-3), "unit": "samples/s",
               "ms_per_step": t.item() / Kb, "steps": Kb, "note": "separate line, not the headline: accuracy 1e-3..1e-2 vs the oracle (tests/test_bf16_mode_gpu.py)"}
        if not a.no_rollout:
            with torch.no_grad():
                for _ in range(3):
                    agent.actor(obs)
                barrier()
                evr = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
                for i in range(5):
                    flush.zero_()
                    evr[i][0].record(); agent.actor(obs); evr[i][1].record()
                barrier()
                t = torch.tensor([sum(s.elapsed_time(e) for s, e in evr)], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                bfl["rollout_limb_tokens_per_s"] = world * a.rollout_envs * N * 5 / (t.item() * 1e-3)
        line["bf16_input_mode"] = bfl
        for m in mods:
            m.use_tc = use_tc

    # ---- reference algorithm on this box's host cores (rank 0, N=1 only; bounded sample)
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cb = cpu_reference_rate(a.morph, B, budget_s=15.0)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "port_over_reference_time") if k in cb}
    if a.check_replicas:
        line["replicas"] = check_replicas(agent, world, dev)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # captured graphs hold NCCL work; tearing the process group down underneath them can hang at exit (seen at N=2):
        # synchronise, meet at a barrier, flush and leave without running destructors
        barrier()
        sys.stdout.flush()
        os._exit(0)


def run_set(a, agent, dev, world, rank, local, init):
    """Multi-morphology step (BASELINE configs "Walker++ multi-morphology update", "cwhh ... sharded across 8 B200"): every
    morphology of the set gets one TD3 update of --batch samples; the set is dealt round-robin over the ranks.  --packed runs a
    rank's morphologies as one packed update; otherwise one update after the other like src/trainer.py:245-250."""
    import torch
    import torch.distributed as dist
    from sgrl_b200 import graph as G, morphologies as M, synth
    names = sorted(M.SETS[a.set])
    mine = names[rank::world]
    B = a.batch
    K, W = a.steps, a.warmup
    # N > 1: the morphologies are dealt over the ranks and every rank runs its share as ONE packed update, so that all ranks
    # issue the same number of gradient all-reduces whatever the split (23 cwhh morphologies over 8 ranks = 3,3,3,3,3,3,3,2);
    # the per-token loss weight uses morph_count = n / world, which makes the all-reduced sum / world the mean over all n
    packed = a.packed or world > 1
    mcount = len(names) / world if world > 1 else None
    if not mine:
        raise SystemExit(f"--set {a.set}: {len(names)} morphologies cannot be dealt over {world} ranks")
    graphs = {n: G.build_graph(M.SETS[a.set][n], device=dev) for n in mine}
    host = {n: {k: v.pin_memory() for k, v in synth.make_batch(B, len(M.SETS[a.set][n]), seed=300 + i).items()} for i, n in enumerate(mine)}
    devb = {n: {k: v.to(dev) for k, v in host[n].items()} for n in mine}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()

    per_morph = {}          # one after the other: the loss dict of every morphology's update in the last step

    def step(i, batches):
        if packed:
            return agent.update_packed([(graphs[n], batches[n]) for n in mine], i, morph_count=mcount)
        ld = None
        for n in mine:
            agent.change_morphology(graphs[n])
            ld = per_morph[n] = agent.update(batches[n], i)
        return ld

    agent.lazy_stats = True
    it = 0
    for _ in range(4 + W):       # 4 set-up steps (eager + graph capture per plan and kind of step), then W warm-up steps
        step(it, devb); it += 1
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for i in range(K):
        restore(agent, init)
        flush.zero_()
        ev[i][0].record(); ld = step(it, devb); it += 1; ev[i][1].record()
    barrier()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, ld if packed else {f"{n}/{k}": v for n, d in per_morph.items() for k, v in d.items()}, agent)
    t = torch.tensor([sum(s.elapsed_time(e) for s, e in ev)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    agent.lazy_stats = False
    for _ in range(4):
        step(it, host)["loss/critic_loss"].item(); it += 1
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        step(it, host)["loss/critic_loss"].item(); it += 1
    barrier()
    t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    nsamp = B * len(names)
    toks = B * sum(len(M.SETS[a.set][n]) for n in names)
    line = {"metric": "SET TD3 update samples/sec", "value": nsamp * K / (total_ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 (3xTF32 tensor-core projections, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": f"{a.set}: {len(names)} morphologies x B={B}, one TD3 update each per step, "
                                   + ("packed into one update per rank (Agent.update_packed)" if packed else "one after the other (src/trainer.py:245-250)"),
                       "morphologies_per_rank": len(mine), "limb_tokens_per_step": toks, "l2": "256 MiB buffer written between timed steps"},
            "e2e": {"value": nsamp * K / t.item(), "unit": "samples/s", "h2d_bytes_per_step": sum(v.numel() * 4 for n in mine for v in host[n].values()),
                    "d2h_bytes_per_step": 4, "how": "update(_packed) with pinned host batches + critic_loss.item(), wall clock, max over ranks"},
            "whole_step_tflops": FLOP_PER_TOKEN_UPDATE * toks / (total_ms / K * 1e-3) / 1e12}
    if a.check_replicas:
        line["replicas"] = check_replicas(agent, world, dev)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        barrier(); sys.stdout.flush(); os._exit(0)


def check_replicas(agent, world, dev):
    """Bitwise comparison of every rank's parameter arenas (live and target nets) after the run: data-parallel replicas
    apply the identical all-reduced gradient, so they must stay identical bit for bit (SURVEY.md §4 tier 5)."""
    import torch
    import torch.distributed as dist
    sums = []
    for m in (agent.actor, agent.critic, agent.actor_target, agent.critic_target):
        bits = m.full_arena.view(torch.int32).to(torch.int64)
        sums += [bits.sum(), (bits * torch.arange(1, bits.numel() + 1, device=dev) % 1000003).sum()]
    mine = torch.stack(sums)
    if world == 1:
        return {"identical": True, "ranks": 1}
    allv = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine)
    same = all(bool((v == allv[0]).all()) for v in allv)
    return {"identical": same, "ranks": world, "checksums_rank0": [int(x) for x in allv[0].tolist()]}


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
