"""Host-side layout of variable-length batches (no GPU): offsets, chunk boundaries and batch offsets, per-utterance output views."""
import torch

from edm_tts_b200 import _lib, varlen


def test_offsets():
    assert varlen.offsets([]) == [0]
    assert varlen.offsets([3, 1, 4]) == [0, 3, 4, 8]


def test_plan_chunks_in_order_with_batch_offsets():
    T = list(range(2, 2 + 130))
    P = [i % 3 for i in range(130)]
    chunks = varlen.plan(T, P, 64, batch_offset=7)
    assert [(c.start, c.stop) for c in chunks] == [(0, 64), (64, 128), (128, 130)]
    assert [c.batch_offset for c in chunks] == [7, 71, 135]
    cu = varlen.offsets(T)
    for c in chunks:
        assert c.T == tuple(T[c.start:c.stop]) and c.P == tuple(P[c.start:c.stop])
        assert c.t0 == cu[c.start]
    assert varlen.plan([5], [0], 64) == [varlen.Chunk(0, 1, 0, (5,), (0,), 0)]


def test_plan_rejects_mismatched_lengths():
    import pytest

    with pytest.raises(ValueError):
        varlen.plan([1, 2], [0], 64)


def test_split_blocks_are_views_of_the_packed_output():
    T, Q = [3, 1, 5], 12
    packed = torch.arange(Q * sum(T))
    views = varlen.split_blocks(packed, T, Q)
    assert [tuple(v.shape) for v in views] == [(Q, t) for t in T]
    assert torch.equal(views[1][:, 0], torch.arange(Q * 3, Q * 3 + Q))
    assert torch.equal(views[2][4], torch.arange(Q * 4 + 4 * 5, Q * 4 + 5 * 5))
    views[0][0, 0] = -1
    assert packed[0] == -1  # a view, not a copy
    # equal lengths: the packed layout is the [B, Q, T] layout of a uniform batch
    u = torch.arange(4 * Q * 6)
    assert torch.equal(torch.stack(varlen.split_blocks(u, [6] * 4, Q)), u.view(4, Q, 6))


def test_varlen_symbols_declared():
    for name in ("edm_s2a_workspace_bytes_varlen", "edm_s2a_bind_varlen", "edm_attention_varlen", "edm_conv_module_varlen"):
        assert name in _lib.EXPORTED_SYMBOLS
