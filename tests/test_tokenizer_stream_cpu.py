"""CPU: the plan SoundStream.stream flattens the convolution stacks into -- history rows per convolution, input activation
and residual wiring -- and its refusal of stacks it would not stream correctly."""
import pytest
import torch.nn as nn

# history rows (k - 1 per causal convolution, 0 for the 1 x 1 convolutions, 1 for the transposed convolution)
ENC_HIST = [4] + [2, 0, 2, 0, 2, 0, 3] * 2 + [2]
DEC_HIST = [2] + [1, 2, 0, 2, 0, 2, 0] * 2 + [4]


def _model():
    from frankenstein_b200.vq_brain import SoundStream
    return SoundStream(C=64, D=64, codebook_size=128, n_electrodes=64)


def test_plan_history_rows_and_wiring():
    from frankenstein_b200.vq_brain import _stream_plan
    m = _model()
    enc, dec = _stream_plan(m.encoder), _stream_plan(m.decoder)
    assert [e.hist for e in enc] == ENC_HIST
    assert [e.hist for e in dec] == DEC_HIST
    assert [e.stride for e in enc] == [1] * 7 + [2] + [1] * 6 + [2, 1]
    assert [e.transposed for e in dec] == [False, True] + [False] * 6 + [True] + [False] * 7
    # every convolution but the first of a stack reads ELU(previous output (+ residual))
    assert [e.elu for e in enc] == [False] + [True] * 15 and [e.elu for e in dec] == [False] + [True] * 15
    # the residual of a ResidualUnit is the input of its causal convolution, added where the next convolution reads it
    assert [e.res for e in enc] == [None, None, None, 1, None, 3, None, 5, None, None, 8, None, 10, None, 12, None]
    assert [e.res for e in dec] == [None, None, None, None, 2, None, 4, None, 6, None, None, 9, None, 11, None, 13]


def _modified(change):
    m = _model()
    change(m)
    return m


@pytest.mark.parametrize("change", [
    lambda m: m.encoder.layers.__setitem__(1, nn.ReLU()),                               # another activation
    lambda m: m.encoder.layers.append(nn.ELU()),                                        # stack ends in an activation
    lambda m: m.encoder.layers[2].layers.__setitem__(1, nn.ELU(alpha=0.5)),             # ELU alpha != 1
    lambda m: m.encoder.layers[2].layers.insert(1, nn.ELU()),                           # ELU(ELU(x))
    lambda m: setattr(m.encoder.layers[2].layers[0].layers[0], "dilation", (2,)),       # dilated causal conv
    lambda m: setattr(m.encoder.layers[2].layers[0].layers[0], "padding", (1,)),        # padded conv
    lambda m: setattr(m.decoder.layers[2].layers[0], "stride", (4,)),                   # transposed conv stride 4
    lambda m: m.decoder.layers[4].layers.__setitem__(0, nn.Identity()),                 # unknown module
    lambda m: m.encoder.layers[2].layers[0].layers.append(nn.ELU()),                    # unit ends in an activation
    lambda m: setattr(m.encoder.layers[4].layers[2], "layers", nn.ModuleList(m.encoder.layers[4].layers[2].layers)),
])
def test_plan_rejects_modified_stacks(change):
    from frankenstein_b200._lib import FkError
    from frankenstein_b200.vq_brain import _stream_plan
    m = _modified(change)
    with pytest.raises(FkError):
        _stream_plan(m.encoder)
        _stream_plan(m.decoder)


def test_plan_rejects_subclasses():
    from frankenstein_b200 import vq_brain
    from frankenstein_b200._lib import FkError

    class MyConv(vq_brain.CausalConv1d):
        def forward(self, x):
            return super().forward(x) * 2

    m = _model()
    old = m.encoder.layers[6]
    m.encoder.layers[6] = MyConv(old.in_channels, old.out_channels, kernel_size=3)
    with pytest.raises(FkError):
        vq_brain._stream_plan(m.encoder)


def test_stream_refuses_cpu_models():
    from frankenstein_b200._lib import FkError
    with pytest.raises(FkError):
        _model().stream(1)
