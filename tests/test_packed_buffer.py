"""Host-side checks of the packed gather over several replay buffers (sgrl_b200.buffer.gather_packed_into): index validation
against each buffer's own capacity, part count and device checks.  No GPU needed; the gather itself is in
test_packed_buffer_gpu.py."""
import pytest
import torch

from sgrl_b200.buffer import MAX_PACKED_PARTS, ReplayBuffer, gather_packed_into


def _cpu_buffers():
    bufs = [ReplayBuffer(41 * n, 3 * n, max_buffer_size=cap, device="cpu") for n, cap in ((2, 10), (3, 20))]
    for b in bufs:
        for i in range(5):
            b.add_transition([i] * b.obs_dim, [i] * b.action_dim, [i] * b.obs_dim, float(i), 0.0)
    return bufs


def _outputs(bufs, counts):
    f = lambda n: torch.zeros(n)
    return (f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(c * b.action_dim for c, b in zip(counts, bufs))),
            f(sum(c * b.obs_dim for c, b in zip(counts, bufs))), f(sum(counts)), f(sum(counts)))


def test_indices_are_checked_against_their_own_buffer():
    bufs = _cpu_buffers()
    # 15 is a valid row of the 20-row buffer but not of the 10-row one: the error names the buffer it overflows
    with pytest.raises(IndexError, match="buffer of 10 rows"):
        gather_packed_into(bufs, [[0, 15], [0]], *_outputs(bufs, [2, 1]))
    with pytest.raises(IndexError, match="buffer of 20 rows"):
        gather_packed_into(bufs, [[0, -10], [-21]], *_outputs(bufs, [2, 1]))
    # the single-buffer path raises the same error
    with pytest.raises(IndexError, match="buffer of 10 rows"):
        bufs[0].get_batch([15])
    assert bufs[0]._staged == 0 and bufs[1]._staged == 0           # the gather flushed every buffer first


def test_parts_devices_and_shapes_are_checked():
    bufs = _cpu_buffers()
    with pytest.raises(ValueError, match=f"1 to {MAX_PACKED_PARTS}"):
        gather_packed_into(bufs * 33, [[0]] * 66, *_outputs(bufs * 33, [1] * 66))
    with pytest.raises(ValueError, match="1 to"):
        gather_packed_into([], [], *_outputs([], []))
    with pytest.raises(ValueError, match="index lists"):
        gather_packed_into(bufs, [[0]], *_outputs(bufs, [1, 1]))
    with pytest.raises(ValueError, match="contiguous fp32"):
        gather_packed_into(bufs, [[0], [1, 2]], *_outputs(bufs, [1, 1]))
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="cpu"):
            gather_packed_into(bufs, [[0], [1]], *(t.cuda() for t in _outputs(bufs, [1, 1])))
    else:
        from sgrl_b200._lib import SgrlError
        with pytest.raises(SgrlError, match="CUDA"):                  # no CPU fallback for the data path
            gather_packed_into(bufs, [[0], [1]], *_outputs(bufs, [1, 1]))
