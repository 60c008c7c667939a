"""CPU: the host side of sliding streams -- the band of a LabelMask (validation, the dense rule with 64-bit differences),
the new C entry points' declarations and their rejections before any launch, and the sliding stream's step rules
(no window limit, at most W patches per row and step, patch indices inside int32), each rejection changing nothing."""
import inspect

import pytest
import torch

from tests.test_stream_sessions_cpu import _encoder


def test_band_validation():
    from frankenstein_b200 import ops
    q = torch.zeros(1, 4, dtype=torch.int32)
    for bad in (0, -1, 1.5, "2"):
        with pytest.raises(ops.FkError, match="band"):
            ops.LabelMask(q, band=bad)
    assert ops._check_band(None) is None and ops._check_band(7) == 7 and ops._check_band(2 ** 40) == 2 ** 40
    with pytest.raises(ops.FkError, match="B200"):
        ops.LabelMask(q, band=3)                  # a valid band, then the CPU tensor is refused


def test_dense_band_rule_in_64_bits():
    from frankenstein_b200 import ops
    lo, hi = -2 ** 31, 2 ** 31 - 1
    m = ops.LabelMask.__new__(ops.LabelMask)
    m.qid = torch.tensor([[lo, 0, 5, hi]], dtype=torch.int32)
    m.kid = torch.tensor([[lo, 0, 3, 4, 5, hi]], dtype=torch.int32)
    for band, rows in ((1, [[1, 0, 0, 0, 0, 0], [0, 1, 0, 0, 0, 0], [0, 0, 0, 0, 1, 0], [0, 0, 0, 0, 0, 1]]),
                       (2, [[1, 0, 0, 0, 0, 0], [0, 1, 0, 0, 0, 0], [0, 0, 0, 1, 1, 0], [0, 0, 0, 0, 0, 1]]),
                       (2 ** 32, [[1, 0, 0, 0, 0, 0], [1, 1, 0, 0, 0, 0], [1, 1, 1, 1, 1, 0], [1, 1, 1, 1, 1, 1]]),
                       (None, [[1, 0, 0, 0, 0, 0], [1, 1, 0, 0, 0, 0], [1, 1, 1, 1, 1, 0], [1, 1, 1, 1, 1, 1]])):
        m.band = band
        assert torch.equal(m.dense()[0, 0], torch.tensor(rows, dtype=torch.bool)), band


def test_entry_points_declared_and_reject_before_launch():
    from frankenstein_b200 import _lib
    protos = _lib.parse_header()
    kv = protos["fk_attn_forward_kv_tc"][1]
    assert protos["fk_attn_forward_kv_band_tc"][1] == kv[:-2] + ["long long"] + kv[-2:]
    assert protos["fk_stream_ring_positions"][1][:7] == ["ptr", "ptr", "ptr", "int", "int", "int", "int"]
    L = _lib.lib()
    args = [None] * 5 + [1, 1, 1, 1, 16] + [0] * 8 + [None] * 6 + [1.0, None, None, 1]
    for band in (0, -1, -2 ** 63):
        assert L.fk_attn_forward_kv_band_tc(*args, band, None, None) == -1
        assert b"band" in L.fk_last_error()
    assert L.fk_stream_ring_positions(None, None, None, 1, 1, 1, 1, *([None] * 8), 1, None, None) == -1
    assert b"fk_stream_ring_positions" in L.fk_last_error()


def test_stream_signatures():
    from frankenstein_b200 import brainformer as bf
    assert inspect.signature(bf.Encoder.stream).parameters["sliding"].default is False
    assert inspect.signature(bf.BrainFormer.stream).parameters["sliding"].default is False


def test_sliding_step_rules_change_nothing():
    from frankenstein_b200 import ops
    enc = _encoder()                              # window 8 patches of 16 electrodes = 128 tokens, patch 8 bins
    s = enc.stream(3, sliding=True)
    assert s.sliding and s.window == 8 and s.cap == 256 and s.caches[0].shape[:2] == (3, 256)
    assert s._keys.kid.shape == (3, 256) and bool((s._keys.kid == 2 ** 31 - 1).all())
    x9 = torch.zeros(3, 9 * 8, 16)               # 9 patches: more than W for every row
    with pytest.raises(ops.FkError, match=r"rows \[0, 1, 2\].*at most W = 8"):
        s.step(x9)
    with pytest.raises(ops.FkError, match=r"rows \[1\]"):
        s.step(x9, [8, 9, 0])
    assert s.lengths == [0, 0, 0]
    s._lengths = [10 ** 6, 128, 0]               # far past the window: no length limit
    with pytest.raises(ops.FkError, match="B200"):
        s.step(torch.zeros(3, 8 * 8, 16))         # W patches for every row fit; then the CPU tensor is refused
    last = (2 ** 31 - 1) * 16                     # first token of the last int32 patch index
    s._lengths = [last, last + 16, 0]
    with pytest.raises(ops.FkError, match=r"rows \[1\].*int32"):
        s.step(torch.zeros(3, 8, 16), [1, 1, 1])  # row 0's new patch is the last int32 one; row 1's passes it
    with pytest.raises(ops.FkError, match="B200"):
        s.step(torch.zeros(3, 8, 16), [1, 0, 1])  # row 1 waits: nothing passes int32
    assert s.lengths == [last, last + 16, 0]
