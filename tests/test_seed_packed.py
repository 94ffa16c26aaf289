"""Seed-batched packed updates without a GPU (SeedBatchedAgent.update_packed_per_seed / update_packed_from_buffers_per_seed,
sgrl_b200.buffer.gather_seeds_into): every argument error is a ValueError raised before anything is drawn from the Python /
numpy random streams and before a plan exists, and the seed-batched gather checks its seeds, parts, geometry and indices on
the host.  The update and the gather themselves are in test_seed_packed_gpu.py."""
import random

import numpy as np
import pytest
import torch

from oracle import ref_loader
from sgrl_b200 import graph as G, morphologies as M, synth

HOPPER, WALKER = M.ALL["3d_hopper_5_full"], M.ALL["3d_walker_7_full"]


def _agent(K=2):
    from sgrl_b200.seed_batch import SeedBatchedAgent
    return SeedBatchedAgent(ref_loader.default_args(), list(range(K)))


def _buffer(n, cap=20, rows=5):
    from sgrl_b200.buffer import ReplayBuffer
    buf = ReplayBuffer(41 * n, 3 * n, max_buffer_size=cap, device="cpu")
    b = synth.make_batch(rows, n, seed=n)
    for i in range(rows):
        buf.add_transition(b["obs"][i].numpy(), b["action"][i].numpy(), b["next_obs"][i].numpy(), float(b["reward"][i]),
                           float(b["done"][i]))
    return buf


def _rng_state():
    return random.getstate(), np.random.get_state()[1].tobytes()


def test_update_packed_per_seed_argument_errors():
    sb = _agent(2)
    gh, gw = G.build_graph(HOPPER), G.build_graph(WALKER)
    bh, bw = synth.make_batch(4, len(HOPPER), seed=1), synth.make_batch(4, len(WALKER), seed=2)
    ok = [(gh, bh), (gw, bw)]
    state = _rng_state()
    with pytest.raises(ValueError, match="one per seed"):
        sb.update_packed_per_seed([ok], 0)
    with pytest.raises(ValueError, match="one per seed"):
        sb.update_packed_per_seed([ok, ok, ok], 0)
    with pytest.raises(ValueError, match="seed 1 morphology 0 has other parents"):
        sb.update_packed_per_seed([ok, [(gw, bw), (gh, bh)]], 0)
    with pytest.raises(ValueError, match="seed 1 has 1 morphologies"):
        sb.update_packed_per_seed([ok, ok[:1]], 0)
    with pytest.raises(ValueError, match="seed 1 morphology 1: a batch of 6 samples"):
        sb.update_packed_per_seed([ok, [(gh, bh), (gw, synth.make_batch(6, len(WALKER), seed=3))]], 0)
    with pytest.raises(ValueError, match="1 to 64 morphologies"):
        sb.update_packed_per_seed([[(gh, bh)] * 65] * 2, 0)
    with pytest.raises(ValueError, match="1 to 64 morphologies"):
        sb.update_packed_per_seed([[], []], 0)
    nz = [torch.zeros(4, 3 * len(HOPPER)), torch.zeros(4, 3 * len(WALKER))]
    with pytest.raises(ValueError, match="noises: expected one per seed"):
        sb.update_packed_per_seed([ok, ok], 0, noises=[nz])
    with pytest.raises(ValueError, match="seed 1 has 1 tensors for 2 morphologies"):
        sb.update_packed_per_seed([ok, ok], 0, noises=[nz, nz[:1]])
    assert _rng_state() == state and len(sb._plans) == 0 and len(sb._packed_tables) == 0


def test_update_packed_from_buffers_per_seed_argument_errors():
    from sgrl_b200.buffer import ReplayBuffer
    sb = _agent(2)
    gh, gw = G.build_graph(HOPPER), G.build_graph(WALKER)
    parts = [[(gh, _buffer(len(HOPPER))), (gw, _buffer(len(WALKER)))] for _ in range(2)]
    state = _rng_state()
    with pytest.raises(ValueError, match="one per seed"):
        sb.update_packed_from_buffers_per_seed(parts[:1], 4, 0)
    with pytest.raises(ValueError, match="seed 1 morphology 0 has other parents"):
        sb.update_packed_from_buffers_per_seed([parts[0], parts[1][::-1]], 4, 0)
    with pytest.raises(ValueError, match="seed 1 buffer 1 rows .* do not match its morphology"):
        sb.update_packed_from_buffers_per_seed([parts[0], [parts[1][0], (gw, _buffer(len(HOPPER)))]], 4, 0)
    empty = ReplayBuffer(41 * len(WALKER), 3 * len(WALKER), max_buffer_size=8, device="cpu")
    with pytest.raises(ValueError, match="seed 0 buffer 1 is empty"):
        sb.update_packed_from_buffers_per_seed([[parts[0][0], (gw, empty)], parts[1]], 4, 0)
    with pytest.raises(ValueError, match="1 to 64 morphologies"):
        sb.update_packed_from_buffers_per_seed([parts[0][:1] * 65] * 2, 4, 0)
    with pytest.raises(ValueError, match="noises: expected one per seed"):
        sb.update_packed_from_buffers_per_seed(parts, 4, 0, noises=[[None, None]])
    if torch.cuda.is_available():                      # the agent's modules sit on the GPU: a CPU buffer is refused
        with pytest.raises(ValueError, match="cpu"):
            sb.update_packed_from_buffers_per_seed(parts, 4, 0)
    assert _rng_state() == state and len(sb._plans) == 0 and len(sb._packed_tables) == 0


def test_single_agent_entry_points_name_the_seed_batched_ones():
    sb = _agent(2)
    for f in (sb.update_packed, sb.update_packed_from_buffers):
        with pytest.raises(NotImplementedError, match="update_packed_per_seed"):
            f([], 0)


def _outputs(bufs_per_seed, counts_per_seed):
    bufs = [b for s in bufs_per_seed for b in s]
    counts = [c for s in counts_per_seed for c in s]
    f = lambda n: torch.zeros(n)
    return (f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(c * b.action_dim for c, b in zip(counts, bufs))),
            f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(counts)), f(sum(counts)))


def test_gather_seeds_into_host_checks():
    from sgrl_b200.buffer import MAX_SEEDS, gather_seeds_into
    seeds = [[_buffer(2, cap=10), _buffer(3, cap=20)], [_buffer(2, cap=30), _buffer(3, cap=10)]]
    idx = [[[0, 1], [2]], [[3, 4], [0]]]
    with pytest.raises(ValueError, match=f"1 to {MAX_SEEDS} seeds"):
        gather_seeds_into(seeds * 5, idx * 5, *_outputs(seeds * 5, [[2, 1]] * 10))
    with pytest.raises(ValueError, match=f"1 to {MAX_SEEDS} seeds"):
        gather_seeds_into([], [], *_outputs([], []))
    with pytest.raises(ValueError, match="1 to 64 buffers"):
        gather_seeds_into([seeds[0] * 33], [[[0]] * 66], *_outputs([seeds[0] * 33], [[1] * 66]))
    with pytest.raises(ValueError, match="seed 1 has 1 buffers"):
        gather_seeds_into([seeds[0], seeds[1][:1]], [idx[0], idx[1][:1]], *_outputs(seeds, [[2, 1], [2]]))
    with pytest.raises(ValueError, match="seed 1 buffer 0 holds rows of 123 obs"):
        gather_seeds_into([seeds[0], seeds[1][::-1]], idx, *_outputs(seeds, [[2, 1], [2, 1]]))
    with pytest.raises(ValueError, match="seed 1 draws 1 rows from buffer 0"):
        gather_seeds_into(seeds, [idx[0], [[3], [0]]], *_outputs(seeds, [[2, 1], [1, 1]]))
    with pytest.raises(ValueError, match="seeds of index lists"):
        gather_seeds_into(seeds, idx[:1], *_outputs(seeds, [[2, 1], [2, 1]]))
    with pytest.raises(ValueError, match="contiguous fp32"):
        gather_seeds_into(seeds, idx, *_outputs(seeds, [[2, 1], [2, 2]]))
    # each index against its own buffer: 15 is a row of seed 1's 30-row buffer 0, not of seed 0's 10-row one
    with pytest.raises(IndexError, match="buffer of 10 rows"):
        gather_seeds_into(seeds, [[[0, 15], [2]], [[15, 4], [0]]], *_outputs(seeds, [[2, 1], [2, 1]]))
    with pytest.raises(IndexError, match="buffer of 10 rows"):
        gather_seeds_into(seeds, [[[0, 1], [19]], [[3, 4], [-11]]], *_outputs(seeds, [[2, 1], [2, 1]]))
    assert all(b._staged == 0 for s in seeds for b in s)              # every buffer was flushed first
    if not torch.cuda.is_available():
        from sgrl_b200._lib import SgrlError
        with pytest.raises(SgrlError, match="CUDA"):                  # no CPU fallback for the data path
            gather_seeds_into(seeds, idx, *_outputs(seeds, [[2, 1], [2, 1]]))
