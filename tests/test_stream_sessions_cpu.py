"""CPU: the host side of streams whose batch rows are independent sessions -- row validation of a per-row reset, per-row
lengths, `length` while the rows agree, and a capacity check that names the rows and changes nothing."""
import pytest
import torch


def _encoder():
    from frankenstein_b200 import brainformer as bf
    cfg = dict(window_size=64, n_electrodes=16, patch_size=8, dim=64, n_layers=1, head_dim=32, hidden_dim=128, n_heads=2,
               n_kv_heads=2)
    return bf.Encoder(bf.MAEConfig(**cfg))


def test_stream_rows_validation():
    from frankenstein_b200 import ops
    assert ops.stream_rows([2, 0], 3, "t") == [2, 0]
    assert ops.stream_rows((), 3, "t") == []
    assert ops.stream_rows(torch.tensor([1]), 3, "t") == [1]
    for bad in ([3], [-1], [0, 0], [1.0], ["a"], 5):
        with pytest.raises(ops.FkError):
            ops.stream_rows(bad, 3, "t")


def test_stream_length():
    from frankenstein_b200 import ops
    assert ops.stream_length([32, 32, 32], "t") == 32
    with pytest.raises(ops.FkError, match="lengths"):
        ops.stream_length([32, 0, 32], "t")


def test_encoder_stream_reset_rows_host_state():
    from frankenstein_b200 import ops
    s = _encoder().stream(3)
    assert s.lengths == [0, 0, 0] and s.length == 0
    for bad in ([3], [0, 0], [-1], [0, 7]):
        with pytest.raises(ops.FkError):
            s.reset(bad)
        assert not s._ragged and s.lengths == [0, 0, 0]
    s.reset([])                                   # nothing to reset: still the lockstep path
    assert not s._ragged
    s.reset([1])
    assert s._ragged and s.lengths == [0, 0, 0] and s.length == 0
    s._lengths = [32, 0, 16]                      # (as steps would leave them)
    with pytest.raises(ops.FkError, match="lengths"):
        s.length
    assert s.lengths == [32, 0, 16]
    s.reset()
    assert not s._ragged and s.length == 0


def test_encoder_stream_capacity_names_rows():
    from frankenstein_b200 import ops
    s = _encoder().stream(3)
    s.reset([0])
    s._lengths = [96, 0, 112]
    with pytest.raises(ops.FkError, match=r"rows \[0, 2\]"):
        s.step(torch.zeros(3, 24, 16))            # 3 patches = 48 tokens: rows 0 and 2 would pass the 128-token window
    assert s.lengths == [96, 0, 112]
    with pytest.raises(ops.FkError, match="B200"):
        s.step(torch.zeros(3, 8, 16))             # fits every row; a CPU tensor is refused next
    assert s.lengths == [96, 0, 112]
