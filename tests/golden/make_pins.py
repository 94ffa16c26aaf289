"""Generate tests/golden/pins.npz: vectors recorded from THIS repository's host code, not from the reference.

    python tests/golden/make_pins.py

set_golden.npz holds what the unmodified reference computed; these pins cover host code that it does not:

* sgrl_b200.graph.build_graph (traversal ranks and relation tensor) for every morphology of sgrl_b200.morphologies.ALL;
  set_golden.npz holds the reference's getGraphDict output for five of them;
* oracle.replay_oracle.ReplayOracle (the restatement of the reference's ReplayBuffer that the device buffer is checked
  against): its storage after 90 transitions into 37 slots, three seeded sample() calls and one get_batch().

tests/test_graph.py and tests/test_buffer.py compare against them, so a change to either is seen even where the
reference is not available.
"""
from __future__ import annotations

import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.replay_oracle import ReplayOracle  # noqa: E402
from sgrl_b200 import graph as G, morphologies as M  # noqa: E402

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pins.npz")
OD, AD, CAP, ADDS = 41 * 3, 3 * 3, 37, 90
SAMPLE_KWS = ({}, {"sequential": True}, {"allow_duplicate": True})
BATCH_IDX = [0, 5, 36, 5]


def transitions(n, seed):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        yield (rng.standard_normal(OD).astype(np.float32), rng.uniform(-1, 1, AD).astype(np.float32),
               rng.standard_normal(OD).astype(np.float32), float(rng.standard_normal()), float(rng.random() < 0.1))


def buffer_draws(buf):
    """{key: array} of the buffer scenario: storage after ADDS transitions, three seeded samples, one get_batch."""
    for t in transitions(ADDS, seed=5):
        buf.add_transition(*t)
    out = {f"buffer/storage/{k}": getattr(buf, k + "_buffer") for k in ("obs", "action", "next_obs", "reward", "done")}
    out["buffer/curr"] = np.array([buf.curr, buf.max_sample_size])
    for i, kw in enumerate(SAMPLE_KWS):
        random.seed(3); np.random.seed(4)
        for k, v in buf.sample(16, **kw).items():
            out[f"buffer/sample{i}/{k}"] = np.asarray(v)
    for k, v in buf.get_batch(BATCH_IDX).items():
        out[f"buffer/get_batch/{k}"] = np.asarray(v)
    return out


def main():
    d = {}
    for name, par in M.ALL.items():
        g = G.build_graph(par)
        d[f"graph/{name}/traversals"] = np.stack([t.numpy() for t in g["traversals"]])
        d[f"graph/{name}/relation"] = g["relation"].numpy()
    d.update(buffer_draws(ReplayOracle(OD, AD, CAP)))
    np.savez_compressed(PATH, **d)
    print(f"wrote {PATH}: {len(d)} arrays, {os.path.getsize(PATH)} bytes")


if __name__ == "__main__":
    main()
