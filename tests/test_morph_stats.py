"""Per-morphology statistics of packed updates without a GPU: the (P,4) part table that make_packed_tables builds for ragged
parts, and the refusals of sgrl_td3_part_stats, which return before anything is launched or written.  The kernel and the
agents' "per_morphology" lists are in test_morph_stats_gpu.py."""
import ctypes

import pytest
import torch

from sgrl_b200 import graph as G, morphologies as M

RAGGED = [("3d_walker_2_right_leg_left_knee", 5), ("3d_humanoid_9_full", 1), ("3d_cheetah_14_full", 3), ("3d_hopper_5_full", 7)]


def test_part_table_of_ragged_parts():
    from sgrl_b200.modules import make_packed_tables
    specs = [(G.build_graph(M.ALL[name]), B) for name, B in RAGGED]
    for morph_count in (None, 2.0 * len(specs)):
        tb = make_packed_tables(specs, "cpu", morph_count)
        want, t0, g0 = [], 0, 0
        for name, B in RAGGED:
            n = len(M.ALL[name])
            want.append([t0, t0 + B * n, g0, g0 + B])
            t0, g0 = t0 + B * n, g0 + B
        assert tb.part_table.dtype == torch.int32 and tb.part_table.is_contiguous()
        assert tb.part_table.tolist() == want == [list(p[:4]) for p in tb.parts]
        assert (tb.T, tb.G) == (t0, g0)
        # each part's tokens map to its own graphs
        for t_a, t_b, g_a, g_b in want:
            assert tb.tok_graph[t_a:t_b].min().item() == g_a and tb.tok_graph[t_a:t_b].max().item() == g_b - 1


def test_single_part_table():
    from sgrl_b200.modules import make_packed_tables
    tb = make_packed_tables([(G.build_graph(M.ALL["3d_humanoid_9_full"]), 4)], "cpu")
    assert tb.part_table.tolist() == [[0, 36, 0, 4]]


def test_refusals_write_nothing():
    """P outside 1..64, K outside 1..8, T or G <= 0 and a NULL required pointer are refused with a negative code and a message;
    the output (host memory here: a refused call never touches it) keeps its contents."""
    from sgrl_b200._lib import lib
    out = (ctypes.c_double * 8)(*([7.0] * 8))
    o = ctypes.addressof(out)
    fake = 256
    n0 = lib.sgrl_launch_count()

    def call(q=fake, target=fake, q1=fake, reward=fake, parts=fake, P=2, T=10, G=5, K=1, hp=fake):
        return lib.sgrl_td3_part_stats(q, target, q1, reward, parts, P, T, G, K, hp, o, None)

    cases = [(dict(P=0), b"P must be 1..64"), (dict(P=65), b"P must be 1..64"), (dict(K=0), b"K must be 1..8"),
             (dict(K=9), b"K must be 1..8"), (dict(T=0), b"empty batch"), (dict(G=-1), b"empty batch")]
    cases += [(dict(**{name: None}), b"null pointer") for name in ("q", "target", "reward", "parts", "hp")]
    for kw, msg in cases:
        assert call(**kw) < 0, kw
        assert msg in lib.sgrl_last_error(), (kw, lib.sgrl_last_error())
    assert lib.sgrl_td3_part_stats(fake, fake, fake, fake, fake, 2, 10, 5, 1, fake, None, None) < 0
    assert b"null pointer" in lib.sgrl_last_error()
    assert list(out) == [7.0] * 8
    assert lib.sgrl_launch_count() == n0
