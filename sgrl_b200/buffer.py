"""Device-resident replay buffer — drop-in for the reference ``common.buffer.ReplayBuffer``
(src/common/buffer.py:35-190; SURVEY.md §8f rank 2) on the data path of ``Agent.update``.

The reference keeps five numpy arrays on the host; every TD3 update fancy-indexes all five,
wraps them in tensors and pushes five pageable H2D copies (buffer.py:103-120) — on a B200
that host work costs more than the fused update itself.  Here one transition is ONE packed
fp32 row in HBM, ``[obs | action | next_obs | reward | done]``:

* ``add_transition`` (host numpy in, one call per env step like trainer.py:125/226) writes
  the row into a pinned staging block; full blocks go to HBM as one contiguous async copy
  (two when the ring wraps).  ``add_batch`` takes transitions that are already on the device.
* ``sample`` / ``get_batch`` draw the indices exactly like the reference (``random.sample``,
  ``numpy.random.choice``, ``random.choice`` — same RNG streams, so equal seeds give equal
  batches), send the B int64 indices, and ONE gather kernel (csrc/replay.cuh,
  ``sgrl_replay_gather``) produces the five batch tensors on the device.
* ``gather_into`` gathers straight into caller-owned buffers: ``Agent.update_from_buffer``
  uses it to fill the static inputs of its captured CUDA graph, so a training step is
  index draw -> 2 KB H2D -> gather -> graph replay, with no host synchronisation.
* ``gather_packed_into`` does the same for several buffers at once (one per morphology) in
  one launch, writing the packed layout of a mixed-morphology update
  (``Agent.update_packed_from_buffers``); ``gather_seeds_into`` does it for K seeds' buffers
  (``SeedBatchedAgent.update_packed_from_buffers_per_seed``).

Same constructor, attributes (``curr``, ``max_sample_size``, ``max_buffer_size``, the five
``*_buffer`` arrays as numpy properties for the trainer's snapshot code,
common/trainer.py:262-320) and method names as the reference.  No CPU fallback: storage
may be created on the CPU for host-logic tests, but sampling needs the CUDA library.
"""
from __future__ import annotations

import random
import warnings
from typing import Dict, Optional

import numpy as np
import torch

from ._lib import ReplayPart, check, lib, ptr, stream

MAX_PACKED_PARTS = 64          # SGRL_REPLAY_MAX_PARTS: buffers one packed gather reads (csrc/replay.cuh)
MAX_SEEDS = 8                  # SGRL_REPLAY_MAX_SEEDS: seeds one seed-batched gather reads, MAX_PACKED_PARTS buffers each


def _dim(space) -> int:
    if isinstance(space, (int, np.integer)):
        return int(space)
    shape = getattr(space, "shape", None)
    if shape is None or len(shape) == 0:
        raise NotImplementedError("sgrl_b200.ReplayBuffer stores continuous (Box) observations/actions only; "
                                  "the SET hot path has no discrete-action variant (buffer.py:42-45)")
    return int(shape[0])


def _check_indices(idx: np.ndarray, capacity) -> None:
    """numpy's error for obs_buffer[indices] (the reference fancy-indexes its arrays, buffer.py:103-120) when an index lies
    outside [-capacity, capacity).  capacity: the buffer's row count, or one per index (a gather over several buffers)."""
    bad = (idx >= capacity) | (idx < -capacity)
    if bad.any():
        cap = capacity if np.ndim(capacity) == 0 else capacity[int(np.argmax(bad))]
        raise IndexError(f"index out of bounds for a buffer of {int(cap)} rows")


def check_packed_buffers(buffers, device, owner: str = "") -> None:
    """What a packed gather needs of its buffers: 1..MAX_PACKED_PARTS of them, all with their rows on `device`.  owner: prefix
    of the messages (the seed the buffers belong to)."""
    if not 1 <= len(buffers) <= MAX_PACKED_PARTS:
        raise ValueError(f"a packed gather reads 1 to {MAX_PACKED_PARTS} buffers, got {len(buffers)}")
    for i, buf in enumerate(buffers):
        if buf.rows.device != torch.device(device):
            raise ValueError(f"{owner}buffer {i} keeps its rows on {buf.rows.device}, the batch goes to {device}")


def check_seed_buffers(buffers_per_seed, device) -> None:
    """What a seed-batched packed gather needs: 1..MAX_SEEDS seeds, each with the same number (1..MAX_PACKED_PARTS) of buffers
    on `device`, buffer i of every seed holding rows of the geometry of seed 0's buffer i."""
    K = len(buffers_per_seed)
    if not 1 <= K <= MAX_SEEDS:
        raise ValueError(f"a seed-batched gather reads 1 to {MAX_SEEDS} seeds, got {K}")
    first = buffers_per_seed[0]
    for k, bufs in enumerate(buffers_per_seed):
        check_packed_buffers(bufs, device, f"seed {k} ")
        if len(bufs) != len(first):
            raise ValueError(f"seed {k} has {len(bufs)} buffers, seed 0 has {len(first)}: every seed reads one per morphology")
        for i, (b, b0) in enumerate(zip(bufs, first)):
            if (b.obs_dim, b.action_dim) != (b0.obs_dim, b0.action_dim):
                raise ValueError(f"seed {k} buffer {i} holds rows of {b.obs_dim} obs / {b.action_dim} action floats, seed 0's "
                                 f"buffer {i} rows of {b0.obs_dim} / {b0.action_dim}")


def _gather_parts(what, launch, buffers, indices, obs, action, next_obs, reward, done, idx_dev) -> int:
    """What every packed gather shares: flush the buffers, check indices[i] against buffers[i]'s own capacity and the outputs'
    sizes, send the concatenated indices (unless idx_dev already holds them), fill one descriptor per buffer and
    launch(desc, idx_dev).  Returns the number of rows gathered."""
    if len(indices) != len(buffers):
        raise ValueError(f"{len(buffers)} buffers, {len(indices)} index lists")
    for buf in buffers:
        buf.flush()
    flat = [np.asarray(ix, dtype=np.int64).reshape(-1) for ix in indices]
    counts = [x.size for x in flat]
    flat = np.concatenate(flat)
    _check_indices(flat, np.repeat(np.array([b.max_buffer_size for b in buffers], dtype=np.int64), counts))
    G = flat.size
    need = ((obs, sum(c * b.obs_dim for c, b in zip(counts, buffers))), (action, sum(c * b.action_dim for c, b in zip(counts, buffers))),
            (next_obs, sum(c * b.obs_dim for c, b in zip(counts, buffers))), (reward, G), (done, G))
    for t, n in need:
        if t.numel() != n or not t.is_contiguous() or t.dtype != torch.float32:
            raise ValueError(f"{what}: expected a contiguous fp32 buffer of {n} floats, got {tuple(t.shape)}")
    if idx_dev is None:
        idx_dev = torch.from_numpy(flat)
        if obs.device.type == "cuda":
            idx_dev = idx_dev.pin_memory()          # torch's caching host allocator, as in ReplayBuffer._indices_to_device
        idx_dev = idx_dev.to(obs.device, non_blocking=True)
    elif idx_dev.numel() != G or idx_dev.dtype != torch.int64 or idx_dev.device != obs.device or not idx_dev.is_contiguous():
        raise ValueError(f"idx_dev: expected {G} contiguous int64 indices on {obs.device}")
    if G == 0:
        return 0
    desc = (ReplayPart * len(buffers))()
    for d, b, c in zip(desc, buffers, counts):
        d.rows, d.row_floats, d.capacity = ptr(b.rows), b.row_floats, b.max_buffer_size
        d.obs_dim, d.act_dim, d.batch = b.obs_dim, b.action_dim, c
    launch(desc, idx_dev)
    return G


def gather_packed_into(buffers, indices, obs, action, next_obs, reward, done, idx_dev=None) -> int:
    """rows of several buffers -> one packed batch, in ONE gather launch (``sgrl_replay_gather_packed``).  indices[i] are the
    row numbers drawn from buffers[i]; the outputs are contiguous fp32 device buffers holding the parts' batches one after the
    other: obs / next_obs sum(B_i * obs_dim_i) floats, action sum(B_i * action_dim_i), reward / done sum(B_i).  With
    obs_dim = 41 N and action_dim = 3 N that is the packed token layout of ``Agent.update_packed``.  idx_dev: a device int64
    tensor that already holds the concatenated indices (a caller with its own upload); otherwise they are sent from pinned
    memory here.  Returns the number of rows gathered."""
    check_packed_buffers(buffers, obs.device)
    outs = (obs, action, next_obs, reward, done)

    def launch(desc, idx):
        check(lib.sgrl_replay_gather_packed(desc, len(buffers), ptr(idx), *(ptr(t) for t in outs), stream()), "sgrl_replay_gather_packed")

    return _gather_parts("gather_packed_into", launch, buffers, indices, *outs, idx_dev)


def gather_seeds_into(buffers_per_seed, indices_per_seed, obs, action, next_obs, reward, done, idx_dev=None) -> int:
    """``gather_packed_into`` of K seeds' buffers in ONE launch (``sgrl_replay_gather_seeds``): buffers_per_seed[k][i] is seed
    k's buffer of morphology i and indices_per_seed[k][i] the rows drawn from it.  Every seed reads the same number of rows
    from its buffer i, of the same geometry, so the outputs hold seed after seed one packed batch each, seed k's at k times
    the per-seed totals: the input layout of ``SeedBatchedAgent.update_packed_per_seed``.  idx_dev as in gather_packed_into
    (all seeds' indices, seed-major).  Returns the number of rows gathered."""
    check_seed_buffers(buffers_per_seed, obs.device)
    K, P = len(buffers_per_seed), len(buffers_per_seed[0])
    if len(indices_per_seed) != K:
        raise ValueError(f"{K} seeds of buffers, {len(indices_per_seed)} seeds of index lists")
    for k, ixs in enumerate(indices_per_seed):
        if len(ixs) != P:
            raise ValueError(f"seed {k}: {P} buffers, {len(ixs)} index lists")
        for i, ix in enumerate(ixs):
            if np.size(ix) != np.size(indices_per_seed[0][i]):
                raise ValueError(f"seed {k} draws {np.size(ix)} rows from buffer {i}, seed 0 {np.size(indices_per_seed[0][i])}: every "
                                 f"seed needs the same batch size per morphology")
    buffers = [b for bufs in buffers_per_seed for b in bufs]
    outs = (obs, action, next_obs, reward, done)

    def launch(desc, idx):
        check(lib.sgrl_replay_gather_seeds(desc, len(buffers), K, ptr(idx), *(ptr(t) for t in outs), stream()), "sgrl_replay_gather_seeds")

    return _gather_parts("gather_seeds_into", launch, buffers, [ix for ixs in indices_per_seed for ix in ixs], *outs, idx_dev)


class ReplayBuffer(object):
    STAGE_ROWS = 1024

    def __init__(self, obs_space, action_space, max_buffer_size=1000000, modular=False, device=None, **kwargs):
        self.max_buffer_size = int(max_buffer_size)
        self.curr = 0
        self.obs_space, self.action_space = obs_space, action_space
        self.obs_dim = _dim(obs_space)
        self.action_dim = _dim(action_space)
        if modular:
            self.action_dim += 3                                   # buffer.py:49-50
        self.discrete_action = False
        self.max_sample_size = 0
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        self.device = torch.device(device)
        od, ad = self.obs_dim, self.action_dim
        self.row_floats = 2 * od + ad + 2
        self._cols = {"obs": (0, od), "action": (od, od + ad), "next_obs": (od + ad, 2 * od + ad),
                      "reward": (2 * od + ad, 2 * od + ad + 1), "done": (2 * od + ad + 1, 2 * od + ad + 2)}
        self.rows = torch.zeros(self.max_buffer_size, self.row_floats, dtype=torch.float32, device=self.device)
        n_stage = max(1, min(self.STAGE_ROWS, self.max_buffer_size))
        pin = self.device.type == "cuda"
        self._stage = [torch.zeros(n_stage, self.row_floats, dtype=torch.float32, pin_memory=pin) for _ in range(2)]
        self._stage_np = [s.numpy() for s in self._stage]
        self._stage_ev = [None, None]       # copy-complete event of each staging block (its pinned memory is reused)
        self._cur_stage, self._staged, self._stage_start = 0, 0, 0

    # ------------------------------------------------------------------ writes
    def clear(self):
        self.flush()
        self.max_sample_size = 0
        self.curr = 0

    def add_traj(self, obs_list, action_list, next_obs_list, reward_list, done_list):
        for obs, action, next_obs, reward, done in zip(obs_list, action_list, next_obs_list, reward_list, done_list):
            self.add_transition(obs, action, next_obs, reward, done)

    def add_transition(self, obs, action, next_obs, reward, done):
        """buffer.py:75-84.  Host values in; the row reaches HBM with the next flush (automatic before sampling)."""
        if self._staged == 0:
            self._stage_start = self.curr
            ev = self._stage_ev[self._cur_stage]
            if ev is not None:
                ev.synchronize()
                self._stage_ev[self._cur_stage] = None
        row = self._stage_np[self._cur_stage][self._staged]
        c = self._cols
        row[c["obs"][0]:c["obs"][1]] = obs
        row[c["action"][0]:c["action"][1]] = action
        row[c["next_obs"][0]:c["next_obs"][1]] = next_obs
        row[c["reward"][0]] = reward
        row[c["done"][0]] = done
        self._staged += 1
        self.curr = (self.curr + 1) % self.max_buffer_size
        self.max_sample_size = min(self.max_sample_size + 1, self.max_buffer_size)
        if self._staged == self._stage[0].shape[0]:
            self.flush()

    def flush(self):
        """Staged rows -> HBM: one contiguous async copy from pinned memory (two when the ring wraps)."""
        n = self._staged
        if n == 0:
            return
        src, start, cap = self._stage[self._cur_stage], self._stage_start, self.max_buffer_size
        first = min(n, cap - start)
        self.rows[start:start + first].copy_(src[:first], non_blocking=True)
        if first < n:
            self.rows[:n - first].copy_(src[first:n], non_blocking=True)
        if self.device.type == "cuda":
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            self._stage_ev[self._cur_stage] = ev
        self._cur_stage ^= 1
        self._staged = 0

    def add_batch(self, obs, action, next_obs, reward, done):
        """n transitions that already live on the device (vectorised envs): rows are assembled there and written
        with one scatter launch (``sgrl_replay_scatter``)."""
        self.flush()
        n = int(obs.shape[0])
        if n > self.max_buffer_size:
            raise ValueError("more transitions than the buffer holds")
        f = lambda x, w: torch.as_tensor(x, dtype=torch.float32, device=self.device).reshape(n, w)
        staged = torch.cat([f(obs, self.obs_dim), f(action, self.action_dim), f(next_obs, self.obs_dim), f(reward, 1), f(done, 1)], dim=1).contiguous()
        dst = ((torch.arange(n, dtype=torch.int64) + self.curr) % self.max_buffer_size)
        dst = (dst.pin_memory() if self.device.type == "cuda" else dst).to(self.device, non_blocking=True)
        check(lib.sgrl_replay_scatter(ptr(self.rows), self.row_floats, self.max_buffer_size, ptr(dst), ptr(staged), n, stream()), "sgrl_replay_scatter")
        self.curr = (self.curr + n) % self.max_buffer_size
        self.max_sample_size = min(self.max_sample_size + n, self.max_buffer_size)

    # ------------------------------------------------------------------ reads
    def draw_indices(self, batch_size, sequential=False, allow_duplicate=False):
        """The reference's index draw, verbatim semantics and RNG streams (buffer.py:87-101)."""
        if not allow_duplicate:
            if batch_size > self.max_sample_size:
                warnings.warn("Sampling larger than buffer size")
            batch_size = min(self.max_sample_size, batch_size)
        if sequential:
            start_index = random.choice(range(self.max_sample_size))
            return [(start_index + i) % self.max_sample_size for i in range(batch_size)]
        if allow_duplicate:
            return np.random.choice(range(self.max_sample_size), batch_size)
        return random.sample(range(self.max_sample_size), batch_size)

    def _indices_to_device(self, indices) -> torch.Tensor:
        if torch.is_tensor(indices) and indices.device == self.device and indices.dtype == torch.int64:
            return indices.contiguous()
        idx = torch.as_tensor(np.asarray(indices), dtype=torch.int64).reshape(-1)
        _check_indices(idx.numpy(), self.max_buffer_size)
        if self.device.type == "cuda":
            idx = idx.pin_memory()          # torch's caching host allocator: no cudaHostAlloc per call, reuse is stream-safe
        return idx.to(self.device, non_blocking=True)

    def gather_into(self, indices, obs, action, next_obs, reward, done):
        """rows[indices] -> the five caller-owned device buffers (contiguous fp32: obs (B,obs_dim) ..., reward (B), done (B))."""
        self.flush()
        idx = self._indices_to_device(indices)
        B = idx.numel()
        for t, w in ((obs, self.obs_dim), (action, self.action_dim), (next_obs, self.obs_dim), (reward, 1), (done, 1)):
            if t.numel() != B * w or not t.is_contiguous() or t.dtype != torch.float32:
                raise ValueError(f"gather_into: expected a contiguous fp32 buffer of {B}x{w}, got {tuple(t.shape)}")
        if B == 0:           # an empty buffer samples an empty batch (buffer.py:88-91 clamps batch_size to max_sample_size)
            return 0
        check(lib.sgrl_replay_gather(ptr(self.rows), self.row_floats, self.max_buffer_size, ptr(idx), B, self.obs_dim, self.action_dim,
                                     ptr(obs), ptr(action), ptr(next_obs), ptr(reward), ptr(done), stream()), "sgrl_replay_gather")
        return B

    def _gather(self, indices) -> Dict[str, torch.Tensor]:
        idx = self._indices_to_device(indices)
        B = idx.numel()
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=self.device)
        out = dict(obs=f(B, self.obs_dim), action=f(B, self.action_dim), next_obs=f(B, self.obs_dim), reward=f(B, 1), done=f(B, 1))
        self.gather_into(idx, out["obs"], out["action"], out["next_obs"], out["reward"], out["done"])
        return out

    def sample(self, batch_size, to_tensor=True, sequential=False, allow_duplicate=False):
        """buffer.py:86-125: dict(obs (B,od), action (B,ad), next_obs, reward (B,1), done (B,1)) — device tensors
        (``to_tensor``) or numpy arrays."""
        out = self._gather(self.draw_indices(batch_size, sequential, allow_duplicate))
        return out if to_tensor else {k: v.cpu().numpy() for k, v in out.items()}

    def get_batch(self, indices, to_tensor=True):
        """buffer.py:127-151.  Like the reference, the tensor form carries reward/done as (B,1,1) (reshape + unsqueeze)."""
        out = self._gather(indices)
        if not to_tensor:
            return {k: v.cpu().numpy() for k, v in out.items()}
        out["reward"] = out["reward"].unsqueeze(1)
        out["done"] = out["done"].unsqueeze(1)
        return out

    # ------------------------------------------------------------------ snapshot interface (common/trainer.py:262-320)
    def _column(self, key):
        self.flush()
        a, b = self._cols[key]
        x = self.rows[:, a:b].cpu().numpy()
        return x.reshape(-1) if key in ("reward", "done") else x

    def _set_column(self, key, value):
        self.flush()
        a, b = self._cols[key]
        v = torch.as_tensor(np.asarray(value), dtype=torch.float32).reshape(-1, b - a)
        if v.shape[0] != self.max_buffer_size:
            raise ValueError(f"{key}_buffer: expected {self.max_buffer_size} rows, got {v.shape[0]}")
        self.rows[:, a:b].copy_(v)

    obs_buffer = property(lambda s: s._column("obs"), lambda s, v: s._set_column("obs", v))
    action_buffer = property(lambda s: s._column("action"), lambda s, v: s._set_column("action", v))
    next_obs_buffer = property(lambda s: s._column("next_obs"), lambda s, v: s._set_column("next_obs", v))
    reward_buffer = property(lambda s: s._column("reward"), lambda s, v: s._set_column("reward", v))
    done_buffer = property(lambda s: s._column("done"), lambda s, v: s._set_column("done", v))

    def resize(self, new_size):
        """buffer.py:153-190."""
        self.flush()
        new_size = int(new_size)
        if new_size == self.max_buffer_size:
            return
        if new_size < self.max_buffer_size:
            self.rows = self.rows[:new_size].clone()
            if self.curr >= new_size:          # buffer has overflowed
                self.curr = 0
                self.max_sample_size = new_size
        else:
            grown = torch.zeros(new_size, self.row_floats, dtype=torch.float32, device=self.device)
            grown[:self.max_buffer_size].copy_(self.rows)
            self.rows = grown
            if self.curr < self.max_sample_size:   # buffer has overflowed
                self.curr = self.max_sample_size
        self.max_buffer_size = new_size
