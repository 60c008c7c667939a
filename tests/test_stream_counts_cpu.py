"""CPU: the host side of per-row counts in a streaming step -- validation of the counts (number, type, range, multiple),
a window check per row with each row's own count, and rejections that name the rows and change nothing."""
import pytest
import torch

from tests.test_stream_sessions_cpu import _encoder


def test_stream_counts_validation():
    from frankenstein_b200 import ops
    assert ops.stream_counts([0, 2, 1], 3, 2, 1, "t") == [0, 2, 1]
    assert ops.stream_counts((8, 0), 2, 8, 4, "t") == [8, 0]
    assert ops.stream_counts(torch.tensor([1, 0]), 2, 2, 1, "t") == [1, 0]
    for bad, match in (([1, 1], "2 counts"), ([1, 1, 1, 1], "4 counts"), ([0, -1, 0], r"rows \[1\]"),
                       ([3, 0, 3], r"rows \[0, 2\]"), ([0, 1.0, 0], "ints"), (None, "ints"), (["a", 0, 0], "ints")):
        with pytest.raises(ops.FkError, match=match):
            ops.stream_counts(bad, 3, 2, 1, "t")
    with pytest.raises(ops.FkError, match=r"rows \[1\].*multiples of 4"):
        ops.stream_counts([4, 6, 0], 3, 8, 4, "t")


def test_encoder_stream_counts_host_state():
    from frankenstein_b200 import ops
    s = _encoder().stream(3)                      # window 8 patches of 16 electrodes = 128 tokens
    x = torch.zeros(3, 16, 16)                    # 2 patches
    for bad in ([1, 1], [0, -1, 0], [0, 3, 0], [0, 1.5, 0]):
        with pytest.raises(ops.FkError):
            s.step(x, bad)
        assert not s._ragged and s.lengths == [0, 0, 0]
    with pytest.raises(ops.FkError, match="B200"):
        s.step(x, [2, 2, 2])                      # full counts: the plain step, which refuses a CPU tensor next
    assert not s._ragged and s.lengths == [0, 0, 0]
    s.reset([0])
    s._lengths = [128, 112, 0]                    # (as steps would leave them)
    with pytest.raises(ops.FkError, match=r"rows \[1\]"):
        s.step(x, [0, 2, 2])                      # row 1 would pass the window; row 0 waits at its end
    assert s.lengths == [128, 112, 0]
    with pytest.raises(ops.FkError, match="B200"):
        s.step(x, [0, 1, 2])                      # every row fits, row 0 with count 0 at the end of its window
    assert s.lengths == [128, 112, 0]
