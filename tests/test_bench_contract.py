"""bench.py's reference arm runs on the CPU (the reference algorithm on the host cores): its JSON line must carry the keys
the driver reads.  (The GPU arm prints the same keys plus roofline / clocks / gpu_launches; it needs a B200.)"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--batch", "8", "--morph", "3d_hopper_3_shin"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "SET TD3 update samples/sec" and line["unit"] == "samples/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["value"] > 0 and line["vs_baseline"] is None
    assert line["config"]["workload"].startswith("3d_hopper_3_shin TD3 Agent.update")
    cb = line["cpu_baseline"]
    from oracle import ref_loader
    # the live reference when it is on this machine (/root/reference/src, baseline/_ref/src, $SGRL_REF), else the oracle port
    assert cb["kind"] == ("reference" if ref_loader.find_reference() else "port")
    assert (cb["kind"] == "reference") == ("port_over_reference_time" in cb)
    assert cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_falls_back_to_the_port_without_the_reference_tree(tmp_path):
    env = dict(os.environ, SGRL_REF="", SGRL_REF_DISABLE="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--batch", "8", "--morph", "3d_hopper_3_shin"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["cpu_baseline"]["kind"] == "port" and line["value"] > 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_is_refused_outside_the_gpu_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)


def _dump(out, *args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "1", "--batch", "32", "--no-cpu-baseline",
                        "--no-rollout", "--no-bf16", "--dump-outputs", str(out), *args],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    files = sorted(os.listdir(out))
    total = 0
    for f in files:
        x = np.load(os.path.join(out, f))
        assert x.dtype in (np.float32, np.float64) and x.ndim == 1 and np.isfinite(x).all(), f
        total += os.path.getsize(os.path.join(out, f))
    assert total <= 64 << 20
    return json.loads(r.stdout.strip().splitlines()[-1]), files


NETS = ["actor_params.npy", "actor_target_params.npy", "critic_params.npy", "critic_target_params.npy"]


@pytest.mark.gpu
def test_gpu_arm_dump_is_the_same_for_the_same_arguments(tmp_path):
    """--dump-outputs: the loss dict of the last of exactly --steps timed updates and a fixed sample of the four networks'
    parameters, float32 / float64 .npy files, 64 MB at most.  Inputs, initial weights and sample positions are seeded: in
    deterministic mode (no order-dependent fp32 atomics) a second run with the same arguments writes the same dump bit for bit."""
    env = dict(os.environ, SGRL_DETERMINISTIC="1")
    line, files = _dump(tmp_path / "a", "--steps", "3", env=env)
    assert line["steps"] == 3
    # 4 set-up + 1 warm-up + 3 timed updates: the last one (it = 7) is a critic-only step, so no actor loss
    assert files == sorted(NETS + ["loss_critic_loss.npy", "misc_train_reward_mean.npy", "misc_train_reward_var.npy"])
    assert np.load(tmp_path / "a" / "loss_critic_loss.npy")[0] > 0
    _, again = _dump(tmp_path / "b", "--steps", "3", env=env)
    assert again == files
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f


@pytest.mark.gpu
def test_gpu_arm_dump_reproduces_to_rounding_in_the_default_mode(tmp_path):
    """Default mode: fp32 atomics change the last bits from run to run, and every timed step starts from the same seeded
    state, so a second run's dump agrees far below the parity bar (one update's worth of summation-order noise)."""
    _, files = _dump(tmp_path / "a", "--steps", "4")
    assert "loss_actor_loss.npy" in files          # the last timed update (it = 8) is an actor step
    _, again = _dump(tmp_path / "b", "--steps", "4")
    assert again == files
    for f in files:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.shape == y.shape and parity.rel_err(x, y) < 1e-5, (f, parity.rel_err(x, y))


@pytest.mark.gpu
def test_gpu_arm_dumps_every_morphology_of_a_sequential_set(tmp_path):
    line, files = _dump(tmp_path, "--steps", "2", "--set", "3d_hoppers")
    assert line["steps"] == 2
    per = ["loss_critic_loss.npy", "loss_actor_loss.npy", "misc_train_reward_mean.npy", "misc_train_reward_var.npy"]
    names = ["3d_hopper_3_shin", "3d_hopper_4_lower_shin", "3d_hopper_5_full"]
    assert files == sorted(NETS + [f"{n}_{f}" for n in names for f in per])
